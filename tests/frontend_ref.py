"""A float64, differentiable restatement of CorrBlock's data path (SURVEY.md Appendix A1-A6 composed as A9), for judging
the fused frontend kernels (build_pyramid, corr_lookup_fused, corr_lookup_fused_backward, build_backward_gauss) and the
training chain at the bench shape.  Written from the appendix and tests/pyref.py, not from the kernels; plain vectorised
torch on any device.  Every quantity is per edge, so callers run it a few edges at a time.

Build (corr.py:61-86, gaussianMask_cuda.py:77-86):
  V = (f1/4)^T (f2/4) in fp64 from the maps' stored values (exact products);
  lvl0 = V + 3 e V_det / den inside the 9 x 9 window at floor(mean) (Q6), e = exp(-(dx^2/cx + dy^2/cy)/2),
  dx = x1 - mean_x; V_det is V DETACHED (GaussianMaskCuda returns no gradient for corr), mean, cov and den carry
  gradients; then 3 x 2x2 average pooling.
Per call (corr.py:88-109):
  m = sigmoid(unbiased 9-tap var(A1 r = 1 on level 1 at coords / 2)), offset[1] <- offset[1] m (Q7, cumulative);
  four r = 3 deformable lookups (A3): x-major taps (Q1), whole tap gated on the top-left corner with x2 / y2 gated on
  their own (Q3), centre tap read as 0 (Q5), F2I saturation and int32 wrap (Q9), no gradient for coords.
Positions: px = fp32(offset + x0), floor, dx = px - floor(px) in fp32; the corner weights are formed in fp32 from dx, dy
(as the samplers form them) and promoted.  Gradients w.r.t. the offsets go through a straight-through position: the
value is the fp32 one, the derivative that of dx = offset + x0 in fp64, so autograd yields A4's offset gradients
(including the centre tap's, which A4 computes at the zeroed position).

Scales.  Every value comes with S = sum |terms| of the same sum, so that an fp32 evaluation of those terms lies within a
small multiple of 2^-24 S of the exact value.  Gradients get their S from a second, "absolute" graph evaluated beside
the first: every nonlinear step y = f(x) is given the surrogate |y| + sum_i |df/dx_i| (xa_i - xa_i.detach()), and every
product the product rule on its operands' scales, so the backward of that graph with |upstream| is the sum of
|chain-rule terms| of each gradient.  A surrogate's value is its quantity's own scale: the levels of the absolute graph
hold the build's S, so a lookup composed with the build is judged against the error its levels carry.  The mask path's
two differences, the variance's v_k - mean and the sigmoid's m (1 - m), are scaled by the sum of their terms, as every
other sum is: their fp32 evaluation is accurate to that, not to their (possibly cancelled) value.

Level-1 positions.  The mask is a few ulps off in fp32, so fp32(coords / 2 + offset[1] m) can round to a neighbouring
float.  Values are continuous in position: `lookup` returns, per level-1 value, how far the sample moves within that
distance (`slack`, as tests/backend_ref.py does).  Gradients are not (offset gradients jump where a position crosses an
integer), so for gradients the caller passes the fp32 post-mask offsets the kernel sampled with (`off1_pos`): the
positions are then identical and only the derivatives come from fp64.
"""
import torch
import torch.nn.functional as F

from backend_ref import _corner_weights, _neighbourhood, f2i, wrap

RADIUS = 3
RD = 2 * RADIUS + 1
TAPS = RD * RD
CENTER = RADIUS * RD + RADIUS
GAUSS_RADIUS = 4


def _taps(r, device):
    k = torch.arange((2 * r + 1) ** 2, device=device)
    return k // (2 * r + 1) - r, k % (2 * r + 1) - r                       # (i - r, j - r) of flat tap (2r+1) i + j (Q1)


def _det(t):
    return None if t is None else t - t.detach()


def _mul(x, xa, y, ya):
    """x * y and its absolute surrogate."""
    v = x * y
    if xa is None and ya is None:
        return v, None
    xs = x.detach().abs() if xa is None else xa.detach()      # a surrogate's value is its quantity's scale
    ys = y.detach().abs() if ya is None else ya.detach()
    a = xs * ys
    if xa is not None:
        a = a + ys * _det(xa)
    if ya is not None:
        a = a + xs * _det(ya)
    return v, a


def _elementwise(fn, xs, xas):
    """y = fn(*xs) for an elementwise fn, and the absolute surrogate |y| + sum |dy/dx_i| (xa_i - xa_i.detach())."""
    y = fn(*xs)
    if all(a is None for a in xas):
        return y, None
    with torch.enable_grad():
        leaves = [x.detach().expand(y.shape).clone().requires_grad_() for x in xs]
        parts = torch.autograd.grad(fn(*leaves).sum(), leaves, allow_unused=True)
    a = y.detach().abs()
    for p, xa in zip(parts, xas):
        if p is not None and xa is not None:
            a = a + p.abs() * _det(xa)
    return y, a


# ------------------------------------------------------------------------------------------------ build
def volume(f1, f2, f1a=None, f2a=None):
    """f1, f2 [e,C,H,W] fp64 -> V [e,P,P] = (f1/4)^T (f2/4), its value scale sum |f1 f2| / 16 and absolute surrogate."""
    a, b = f1.flatten(2) / 4.0, f2.flatten(2) / 4.0
    V = torch.einsum("ecp,ecq->epq", a, b)
    S = torch.einsum("ecp,ecq->epq", a.detach().abs(), b.detach().abs())
    Va = None
    if f1a is not None or f2a is not None:
        Va = S.clone()
        if f1a is not None:
            Va = Va + torch.einsum("ecp,ecq->epq", _det(f1a.flatten(2)) / 4.0, b.detach().abs())
        if f2a is not None:
            Va = Va + torch.einsum("ecp,ecq->epq", a.detach().abs(), _det(f2a.flatten(2)) / 4.0)
    return V, S, Va


def _window(means, H, W):
    """The 9 x 9 window of every pixel at floor(mean) (A5): flat target index [e,P,81] (0 where gated), gate, x1, y1."""
    e = means.shape[0]
    m = means.reshape(e, -1, 1, 2).float()
    ti, tj = _taps(GAUSS_RADIUS, means.device)
    x1 = wrap(f2i(torch.floor(m[..., 0])) + ti)
    y1 = wrap(f2i(torch.floor(m[..., 1])) + tj)
    inb = (x1 >= 0) & (x1 < W) & (y1 >= 0) & (y1 < H)
    idx = torch.where(inb, y1 * W + x1, torch.zeros_like(x1))
    return idx, inb, x1.double(), y1.double()


def build(V, S_V, means, covs, den, H, W, Va=None, means_a=None, covs_a=None, den_a=None, corr_through_gauss=False,
          level3_share=1.0 / 64.0):
    """The Gaussian residual and the 4-level pyramid.  V [e,P,P] fp64 (S_V its value scale); means, covs [e,H,W,2],
    den [e,H,W] fp64.  Returns (levels [4 x [e,P,Q_l]], their value scales, their absolute surrogates or Nones).
    Near misses for the tests' bars: corr_through_gauss lets V's gradient flow through the Gaussian branch;
    level3_share != 1/64 rescales level 3's share of the gradient (its value is unchanged)."""
    e, P, _ = V.shape
    idx, inb, x1, y1 = _window(means, H, W)
    mx, my = means.reshape(e, P, 1, 2)[..., 0], means.reshape(e, P, 1, 2)[..., 1]
    cx, cy = covs.reshape(e, P, 1, 2)[..., 0], covs.reshape(e, P, 1, 2)[..., 1]
    dn = den.reshape(e, P, 1)
    absd = Va is not None or means_a is not None
    mxa = cxa = mya = cya = dna = None
    if absd:
        mxa, mya = means_a.reshape(e, P, 1, 2)[..., 0], means_a.reshape(e, P, 1, 2)[..., 1]
        cxa, cya = covs_a.reshape(e, P, 1, 2)[..., 0], covs_a.reshape(e, P, 1, 2)[..., 1]
        dna = den_a.reshape(e, P, 1)

    def gfac(mx, my, cx, cy, dn):
        ddx, ddy = x1 - mx, y1 - my
        return 3.0 * torch.exp(-0.5 * (ddx * ddx / cx + ddy * ddy / cy)) / dn

    G, Ga = _elementwise(gfac, (mx, my, cx, cy, dn), (mxa, mya, cxa, cya, dna))     # [e,P,81]
    Vsrc = V if corr_through_gauss else V.detach()
    Vw = torch.where(inb, Vsrc.gather(-1, idx), torch.zeros((), dtype=V.dtype, device=V.device))
    Vwa = None
    if absd:                                    # the window's scale; a gradient only through the near miss
        src = S_V if Va is None else (Va if corr_through_gauss else Va.detach())
        Vwa = torch.where(inb, src.gather(-1, idx), torch.zeros((), dtype=V.dtype, device=V.device))
    r, ra = _mul(G, Ga, Vw, Vwa)
    zero = torch.zeros((), dtype=V.dtype, device=V.device)
    r = torch.where(inb, r, zero)
    lvl0 = V + torch.zeros_like(V).scatter_add(-1, idx, r)
    Sw = torch.where(inb, S_V.gather(-1, idx), zero) * G.detach().abs()
    S0 = S_V + torch.zeros_like(S_V).scatter_add(-1, idx, torch.where(inb, Sw, zero))
    lvl0a = None
    if absd:
        base = Va if Va is not None else S_V
        lvl0a = base + torch.zeros_like(V).scatter_add(-1, idx, torch.where(inb, ra, zero))

    def pool(t, l):
        h, w = H >> (l - 1), W >> (l - 1)
        return F.avg_pool2d(t.reshape(e * P, 1, h, w), 2, stride=2).reshape(e, P, -1)

    levels, scales, absl = [lvl0], [S0], [lvl0a]
    for l in range(1, 4):
        nv = pool(levels[-1], l)
        na = pool(absl[-1], l) if absd else None
        if l == 3 and level3_share != 1.0 / 64.0:
            k = level3_share * 64.0 - 1.0
            nv = nv + k * _det(nv)
            na = None if na is None else na + k * _det(na)
        levels.append(nv)
        scales.append(pool(scales[-1], l))
        absl.append(na)
    return levels, scales, absl


# ------------------------------------------------------------------------------------------------ lookup
def _sample(L, La, px, py, sx, sy, sxa, sya, ti, tj, h, w, per_corner=False, swap_dx=False, cnt=None):
    """Bilinear samples of level L [e,P,Q] (fp64; La its absolute surrogate or None) at fp32 positions px, py [e,P,K],
    taps (ti, tj) [K].  sx, sy: the straight-through parts (offset - offset.detach()) or None; sxa, sya likewise for
    the absolute graph.  Returns (values [e,P,K], absolute surrogate, value scale, fxp count term or None).
    Gating: the whole tap on its top-left corner, x2 / y2 on their own (Q3); per_corner: each corner on its own (Q4,
    a near miss).  swap_dx: 1 - dx and dx swapped (a near miss).  cnt [e,P,1]: also return sum over valid corners of
    La * cnt (whose gradient w.r.t. La counts each corner's contribution, weighted by cnt)."""
    e, P, K = px.shape
    fx, fy = torch.floor(px), torch.floor(py)
    x1 = wrap(f2i(fx) + ti)
    y1 = wrap(f2i(fy) + tj)
    dx, dy = px - fx, py - fy                                               # fp32
    if swap_dx:
        dx = 1.0 - dx
    w32 = _corner_weights(dx, dy).double()                                  # [e,P,K,4]
    x2, y2 = wrap(x1 + 1), wrap(y1 + 1)
    cx = torch.stack((x1, x2, x1, x2), -1)
    cy = torch.stack((y1, y1, y2, y2), -1)
    inb = (cx >= 0) & (cx < w) & (cy >= 0) & (cy < h)
    tap = inb[..., 0]
    # a skipped tap has no gradient at all (A4): its fractions must not reach the derivative (a NaN x would, as NaN * 0)
    live = inb.any(-1) if per_corner else tap
    X = torch.where(live, dx.double(), torch.zeros((), dtype=torch.float64, device=dx.device))
    Y = torch.where(live, dy.double(), torch.zeros((), dtype=torch.float64, device=dx.device))
    if sx is not None:
        X = X + (-sx if swap_dx else sx)
        Y = Y + sy
        w64 = torch.stack(((1 - Y) * (1 - X), X * (1 - Y), Y * (1 - X), X * Y), -1)
        wv = w32 + _det(w64)
    else:
        wv = w32
    wa = None
    if La is not None:
        wa = w32.abs()
        if sxa is not None:
            ax = torch.stack(((1 - Y).abs(), (1 - Y).abs(), Y.abs(), Y.abs()), -1).detach()
            ay = torch.stack(((1 - X).abs(), X.abs(), (1 - X).abs(), X.abs()), -1).detach()
            wa = wa + ax * _det(sxa).unsqueeze(-1) + ay * _det(sya).unsqueeze(-1)
    valid = inb if per_corner else inb & tap.unsqueeze(-1)
    flat = torch.where(valid, cy * w + cx, torch.zeros_like(cx)).view(e, P, K * 4)
    zero = torch.zeros((), dtype=torch.float64, device=px.device)
    Q = torch.where(valid, L.gather(-1, flat).view(e, P, K, 4), zero)
    Qa = None if La is None else torch.where(valid, La.gather(-1, flat).view(e, P, K, 4), zero)
    prod, proda = _mul(wv, wa, Q, Qa)
    val = prod.sum(-1)
    S = (w32.abs() * (Q.detach().abs() if Qa is None else Qa.detach())).sum(-1)
    vala = None if proda is None else proda.sum(-1)
    if not per_corner:
        val = torch.where(tap, val, zero)
        S = torch.where(tap, S, zero)
        vala = None if vala is None else torch.where(tap, vala, zero)
    c = None
    if cnt is not None and Qa is not None:
        c = (Qa * cnt.unsqueeze(-1)).sum()
    return val, vala, S, c


def _fp32_position(c, o32):
    return c.unsqueeze(-1) + o32                                            # fp32 add (A3)


def lookup(levels, coords, off0, off1, H, W, levels_a=None, off0_a=None, off1_a=None, off1_pos=None, with_slack=True,
           fxp=None, biased_var=False, drop_mask_grad=False, per_corner=False, swap_dx_level=None):
    """One CorrBlock.__call__ (corr.py:88-109) on an edge chunk.
    levels: 4 fp64 tensors [e,P,Q_l] (H x W source grid, H>>l x W>>l targets); coords [e,P,2] fp32 (level-0 units);
    off0, off1 [e,P,98] fp64: level 0's offsets and offset[1] BEFORE this call's mask; *_a: absolute surrogates or None.
    off1_pos: fp32 [e,P,98] post-mask offsets to take the level-1 positions from (default fp32 of this statement's own).
    fxp [e,P] or None: per-pixel weight whose sum over the valid level-0/1 corners is returned as `fxp` (its gradient
    w.r.t. the absolute levels is the per-element contribution count times that weight).
    Near misses: biased_var, drop_mask_grad (no gradient from the mask into level 1), per_corner (Q4 gating),
    swap_dx_level.
    Returns dict: corr [e,P,196] (+ corr_a), scale, slack (level 1; zero elsewhere), mask [e,P] (+ mask_a, mask_scale),
    off1 (= off1 * mask, + off1_a), fxp."""
    e, P, _ = coords.shape
    dev = coords.device
    absd = levels_a is not None
    out = {}
    # ---- mask: A1 r = 1 on level 1 at coords / 2, unbiased variance of the 9 taps, sigmoid
    c1 = coords / 2.0
    mi, mj = _taps(1, dev)
    L1, L1a = levels[1], (levels_a[1] if absd else None)
    if drop_mask_grad:
        L1, L1a = L1.detach(), (None if L1a is None else L1a.detach())
    px = c1[..., 0:1].expand(e, P, 9).contiguous()
    py = c1[..., 1:2].expand(e, P, 9).contiguous()
    v9, v9a, S9, _ = _sample(L1, L1a, px, py, None, None, None, None, mi, mj, H >> 1, W >> 1)
    n = 9 if biased_var else 8
    mean = v9.mean(-1, keepdim=True)
    var = ((v9 - mean) ** 2).sum(-1) / n
    dv = (v9 - mean).detach()
    S_var = ((2.0 * dv.abs() * S9 + dv * dv) / 8.0).sum(-1)               # value scale of var
    m = torch.sigmoid(var)
    md = m.detach()
    ma = None
    if absd:
        # differences are scaled by the sum of their terms: d var / d v_k = 2 (v_k - mean) / n by S(v_k) + S(mean),
        # d sigmoid = m - m^2 by m + m^2 (an fp32 v_k - mean or 1 - m is accurate to that sum, not to its value)
        dvs = S9 + S9.mean(-1, keepdim=True)
        vara = var.detach().abs() + (2.0 * dvs / n * _det(v9a)).sum(-1)
        ma = md + md * (1 + md) * _det(vara)
    out["mask"], out["mask_a"] = m, ma
    out["mask_scale"] = md * (1 - md) * S_var + md                          # |dm| <= BAR * this
    # ---- offset[1] <- offset[1] * mask (cumulative across calls: the caller chains the returned off1)
    o1, o1a = _mul(off1, off1_a, m.unsqueeze(-1), None if ma is None else ma.unsqueeze(-1))
    out["off1"], out["off1_a"] = o1, o1a
    o1_pos = o1.detach().float() if off1_pos is None else off1_pos
    # ---- four deformable r = 3 lookups
    ti, tj = _taps(RADIUS, dev)
    vals, valsa, scales, slacks, fx_terms = [], [], [], [], []
    for l in range(4):
        h, w = H >> l, W >> l
        cl = coords / float(2 ** l)
        L = levels[l]
        La = levels_a[l] if absd else None
        if l == 0:
            ov, oa, o32 = off0, off0_a, off0.detach().float()
        elif l == 1:
            ov, oa, o32 = o1, o1a, o1_pos
        else:
            ov = oa = None
            o32 = torch.zeros(e, P, 2 * TAPS, dtype=torch.float32, device=dev)
        o32 = o32.reshape(e, P, TAPS, 2).clone()
        o32[:, :, CENTER] = 0.0                                             # Q5: the centre tap reads 0
        px = _fp32_position(cl[..., 0], o32[..., 0])
        py = _fp32_position(cl[..., 1], o32[..., 1])
        sx = sy = sxa = sya = None
        if ov is not None and ov.requires_grad:
            ov2 = ov.reshape(e, P, TAPS, 2)
            sx, sy = _det(ov2[..., 0]), _det(ov2[..., 1])
        if oa is not None:
            oa2 = oa.reshape(e, P, TAPS, 2)
            sxa, sya = _det(oa2[..., 0]), _det(oa2[..., 1])
        cnt = fxp.unsqueeze(-1) if (fxp is not None and l < 2) else None
        v, va, s, c = _sample(L, La, px, py, sx, sy, sxa, sya, ti, tj, h, w, per_corner, swap_dx_level == l, cnt)
        vals.append(v)
        valsa.append(va)
        scales.append(s)
        if c is not None:
            fx_terms.append(c)
        sl = torch.zeros_like(s)
        if l == 1 and with_slack:
            # the position's uncertainty: 1e-6 of the offset (the mask) + 2 ulps of the sum; none for far-out or
            # non-finite positions (their samples are 0 or NaN either way) and for the centre tap
            dlt = []
            for pp, oo in ((px, o32[..., 0]), (py, o32[..., 1])):
                d = 1e-6 * oo.double().abs().clamp(min=1.0) + 2.0 ** -22 * pp.double().abs()
                d = torch.where(torch.isfinite(d) & (pp.double().abs() < 1e6), d, torch.zeros_like(d))
                d[:, :, CENTER] = 0.0
                dlt.append(d)
            with torch.no_grad():
                for qx in _neighbourhood(px, dlt[0]):
                    for qy in _neighbourhood(py, dlt[1]):
                        vq, _, _, _ = _sample(L.detach(), None, qx, qy, None, None, None, None, ti, tj, h, w, per_corner,
                                              swap_dx_level == l)
                        sl = torch.maximum(sl, torch.nan_to_num((vq - v.detach()).abs(), nan=0.0))
        slacks.append(sl)
    out["corr"] = torch.cat(vals, -1)
    out["corr_a"] = torch.cat(valsa, -1) if absd else None
    out["scale"] = torch.cat(scales, -1)
    out["slack"] = torch.cat(slacks, -1)
    out["fxp"] = sum(fx_terms) if fx_terms else None
    return out

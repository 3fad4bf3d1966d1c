"""tests/frontend_ref.py (the float64 statement of CorrBlock's data path that the fused frontend kernels are judged by)
against the CPU oracle's operators composed the way the reference composes them -- corr.py:61-109 and
gaussianMask_cuda.py:7-24,77-86 restated in fp32 torch with oracle/lgu_oracle.c behind every custom operator -- over
three consecutive lookups and one backward, and the bar's power to reject near misses.  Small grids, no GPU.

Bar.  The oracle graph is fp32 throughout; its longest sums (the volume's K = 128 products, the feature-map gradients'
few hundred) are within n 2^-24 sum|terms| <= 2^-15 S of the exact value, so every value and gradient must satisfy
|oracle - fp64| <= BAR S + slack with BAR = 2^-14."""
import pytest
import torch
import torch.nn.functional as F

import frontend_ref as fr
import inputs

BAR = 2.0 ** -14
E, T, C = 2, 4, 128
CALLS = 3


def _ops(orc):
    class Gauss(torch.autograd.Function):                 # gaussianMask_cuda.py:7-24: no gradient for corr
        @staticmethod
        def forward(ctx, mean, cov, corr):
            ctx.save_for_backward(mean, cov, corr)
            return orc.gaussianMask(mean.contiguous(), cov.contiguous(), corr.contiguous(), 4)[0]

        @staticmethod
        def backward(ctx, g):
            mean, cov, corr = ctx.saved_tensors
            gm, gc = orc.gaussianMask_backward(mean.contiguous(), cov.contiguous(), corr.contiguous(), g.contiguous(), 4)
            return gm, gc, None

    class Sampler(torch.autograd.Function):               # corr.py:10-24
        @staticmethod
        def forward(ctx, vol, coords, r):
            ctx.save_for_backward(vol, coords)
            ctx.r = r
            return orc.corr_index_forward(vol.contiguous(), coords.contiguous(), r)[0]

        @staticmethod
        def backward(ctx, g):
            vol, coords = ctx.saved_tensors
            return orc.corr_index_backward(vol.contiguous(), coords.contiguous(), g.contiguous(), ctx.r)[0], None, None

    class DefSampler(torch.autograd.Function):            # corr.py:26-42 (the kernel zeroes the centre taps in place)
        @staticmethod
        def forward(ctx, vol, coords, offset, r):
            off = offset.detach().clone().contiguous()
            out = orc.defCorr_index_forward(vol.contiguous(), coords.contiguous(), off, r)[0]
            ctx.save_for_backward(vol, coords, off)
            ctx.r = r
            return out

        @staticmethod
        def backward(ctx, g):
            vol, coords, off = ctx.saved_tensors
            gv, go = orc.defCorr_index_backward(vol.contiguous(), coords.contiguous(), off.clone(), g.contiguous(), ctx.r)
            return gv, None, go, None

    return Gauss, Sampler, DefSampler


def _case(seed, H, W, nan_probes):
    g = inputs.gen(seed)
    fm = torch.randn(T, C, H, W, generator=g).half().float()
    ii, jj = inputs.edge_list(T, E, g)
    ga = inputs.gaussian_case(E=E, H1=H, W1=W, H2=H, W2=W, seed=seed + 1, probes=True)
    coords = []
    for _ in range(CALLS):
        c = inputs.make_coords(E, H, W, H, W, g, probes=True).permute(0, 2, 3, 1).contiguous()
        if not nan_probes:          # a NaN coordinate makes NaN feature-map gradients everywhere (g_f2 sums all pixels)
            c = torch.nan_to_num(c, nan=-1e10)
        coords.append(c)
    off0 = (4 * torch.tanh(torch.randn(E, H, W, 98, generator=g))).contiguous()
    off1 = ((4 * torch.tanh(torch.randn(E, H, W, 98, generator=g)) + off0) / 2).contiguous()
    wts = [torch.randn(E, 196, H, W, generator=g) for _ in range(CALLS)]
    covs = ga["covs"]
    return dict(f1=fm[ii.long()].contiguous(), f2=fm[jj.long()].contiguous(), means=ga["means"], covs=covs,
                den=(6.28 * torch.sqrt(covs[..., 0] * covs[..., 1])).contiguous(), coords=coords, off0=off0, off1=off1,
                wts=wts, H=H, W=W)


def _oracle_graph(orc, c):
    """The reference's CorrBlock on the oracle's operators, fp32: outputs, masks, post-mask offsets and leaf gradients."""
    Gauss, Sampler, DefSampler = _ops(orc)
    H, W = c["H"], c["W"]
    P = H * W
    leaves = {k: c[k].clone().requires_grad_() for k in ("f1", "f2", "means", "covs", "den", "off0", "off1")}
    f1, f2 = leaves["f1"], leaves["f2"]
    V = torch.matmul(f1.reshape(E, C, P).transpose(1, 2) / 4.0, f2.reshape(E, C, P) / 4.0).view(E, H, W, H, W)
    corr1 = Gauss.apply(leaves["means"], leaves["covs"], V) / leaves["den"].view(E, H, W, 1, 1) + V
    corr1.retain_grad()                                   # the merged level gradient the build's backward consumes
    cur, pyr = corr1.reshape(E * P, 1, H, W), []
    for l in range(4):
        pyr.append(cur.view(E, H, W, H >> l, W >> l))
        if l < 3:
            cur = F.avg_pool2d(cur, 2, stride=2)
    offs = [leaves["off0"], leaves["off1"], torch.zeros(E, H, W, 98), torch.zeros(E, H, W, 98)]
    outs, masks, pos, loss = [], [], [], 0.0
    for k in range(CALLS):
        cc = c["coords"][k].permute(0, 3, 1, 2).contiguous()
        m9 = Sampler.apply(pyr[1], cc / 2, 1)
        m = torch.sigmoid(torch.var(m9.permute(0, 3, 4, 1, 2), dim=[3, 4]))
        offs[1] = offs[1] * m.view(E, H, W, 1)
        masks.append(m.detach())
        pos.append(offs[1].detach().reshape(E, P, 98).clone())
        out = torch.cat([DefSampler.apply(pyr[l], cc / 2 ** l, offs[l].reshape(E, H, W, 7, 7, 2), 3).reshape(E, 49, H, W)
                         for l in range(4)], 1)
        outs.append(out.detach())
        loss = loss + (out * c["wts"][k]).sum()
    loss.backward()
    grads = {k: v.grad for k, v in leaves.items()}
    grads["lvl0"] = corr1.grad.reshape(E, P, P)
    return outs, masks, pos, grads


def _statement(c, pos=None, absolute=True, **knobs):
    """The fp64 statement: values of every call (with slack when pos is None) and, when pos is given (the oracle's
    post-mask offsets), the leaf gradients with their scales."""
    H, W = c["H"], c["W"]
    P = H * W
    names = ("f1", "f2", "means", "covs", "den", "off0", "off1")
    lv = {k: c[k].double().requires_grad_() for k in names}
    la = {k: c[k].double().abs().requires_grad_() for k in names} if absolute else dict.fromkeys(names)
    bk = {k: knobs.pop(k) for k in ("corr_through_gauss", "level3_share") if k in knobs}
    V, S_V, Va = fr.volume(lv["f1"], lv["f2"], la["f1"], la["f2"])
    levels, scales, levels_a = fr.build(V, S_V, lv["means"], lv["covs"], lv["den"], H, W, Va, la["means"], la["covs"],
                                        la["den"], **bk)
    if not absolute:
        levels_a = None
    o0, o0a = lv["off0"].view(E, P, 98), (la["off0"].view(E, P, 98) if absolute else None)
    o1, o1a = lv["off1"].view(E, P, 98), (la["off1"].view(E, P, 98) if absolute else None)
    res, loss, loss_a = [], 0.0, 0.0
    for k in range(CALLS):
        r = fr.lookup(levels, c["coords"][k].view(E, P, 2), o0, o1, H, W, levels_a, o0a, o1a,
                      off1_pos=None if pos is None else pos[k], with_slack=pos is None, **knobs)
        o1, o1a = r["off1"], r["off1_a"]
        w = c["wts"][k].permute(0, 2, 3, 1).reshape(E, P, 196).double()
        loss = loss + (r["corr"] * w).sum()
        if absolute:
            loss_a = loss_a + (r["corr_a"] * w.abs()).sum()
        res.append(r)
    grads = scales_g = None
    if pos is not None:
        grads = dict(zip(names + ("lvl0",), torch.autograd.grad(loss, [lv[k] for k in names] + [levels[0]])))
        if absolute:
            scales_g = dict(zip(names + ("lvl0",), torch.autograd.grad(loss_a, [la[k] for k in names] + [levels_a[0]])))
    return res, levels, scales, grads, scales_g


def _worst(got, ref, scale, slack=None):
    gn, rn = torch.isnan(got), torch.isnan(ref)
    assert torch.equal(gn, rn), f"NaN patterns differ at {int((gn != rn).sum())} values"
    ok = ~rn
    err = (got[ok].double() - ref[ok]).abs()
    if slack is not None:
        err = (err - slack[ok]).clamp(min=0.0)
    s = torch.nan_to_num(scale[ok], nan=0.0)
    ratio = torch.where(err == 0, torch.zeros_like(err), err / s)
    return float(ratio.max()) if ratio.numel() else 0.0


def _flat(t, H, W):
    """[E,196,H,W] -> [E,P,196]."""
    return t.permute(0, 2, 3, 1).reshape(E, H * W, -1)


GRIDS = [(8, 16), (16, 16)]


@pytest.mark.parametrize("grid", GRIDS)
def test_statement_values_match_the_oracle_over_three_calls(oracle, grid):
    """A1/A3 values, the build (A5 + A9's pooling) and the cumulative mask (Q7), NaN / inf / 2^31 / border probes in
    the coordinates and Gaussian means over every border and far outside."""
    H, W = grid
    c = _case(11 + H, H, W, nan_probes=True)
    pyr = oracle.build_pyramid(c["f1"], c["f2"], c["means"], c["covs"])
    outs, masks, _, _ = _oracle_graph(oracle, c)
    with torch.no_grad():
        res, levels, scales, _, _ = _statement(c)
    for l in range(4):
        w = _worst(pyr[l].reshape(E, H * W, -1), levels[l].detach(), scales[l])
        print(f"[frontend ref cpu] {grid} level {l}: worst err/S {w:.3g}")
        assert w <= BAR
    nan_seen = False
    for k in range(CALLS):
        r = res[k]
        w = _worst(_flat(outs[k], H, W), r["corr"].detach(), r["scale"], r["slack"])
        wm = _worst(masks[k].reshape(E, -1), r["mask"].detach(), r["mask_scale"])
        print(f"[frontend ref cpu] {grid} call {k}: corr worst err/S {w:.3g}, mask {wm:.3g}, "
              f"{int((r['slack'] > 0).sum())} values with slack")
        assert w <= BAR and wm <= BAR
        nan_seen |= bool(torch.isnan(outs[k]).any())
    assert nan_seen


@pytest.fixture(scope="module")
def grad_case(oracle):
    H, W = GRIDS[0]
    c = _case(5, H, W, nan_probes=False)
    outs, masks, pos, og = _oracle_graph(oracle, c)
    _, _, _, grads, scales = _statement(c, pos=pos)
    return c, pos, og, grads, scales


def test_statement_gradients_match_the_oracle_graph(grad_case):
    """A2/A4 through autograd (the merged level gradient, offset gradients, the mask path), A6 (means / covs), den, and
    the feature-map gradients of the build, after three cumulative lookups and one backward."""
    c, pos, og, grads, scales = grad_case
    for k in grads:
        w = _worst(og[k].reshape(-1), grads[k].detach().reshape(-1), scales[k].reshape(-1))
        print(f"[frontend ref cpu] grad {k}: worst err/S {w:.3g}")
        assert w <= BAR, k
        assert (og[k] != 0).any()


NEAR_MISSES = [
    ("corr gradient through the Gaussian branch", dict(corr_through_gauss=True)),
    ("biased variance", dict(biased_var=True)),
    ("no mask-path gradient into level 1", dict(drop_mask_grad=True)),
    ("per-corner gating (Q4)", dict(per_corner=True)),
    ("dx and 1 - dx swapped on level 0", dict(swap_dx_level=0)),
    ("dx and 1 - dx swapped on level 2", dict(swap_dx_level=2)),
    ("level 3 weighted 1/16", dict(level3_share=1.0 / 16.0)),
]


@pytest.mark.parametrize("name,knobs", NEAR_MISSES, ids=[n for n, _ in NEAR_MISSES])
def test_the_bar_rejects_near_misses(grad_case, name, knobs):
    """Each near miss, evaluated with the same positions, must exceed the bar somewhere (values or gradients), judged
    against the correct statement's scales, by a margin (4x; the weakest, the mask path's share of level 1, shows ~11x
    at this fp32 bar and ~10^4 x at the kernels' bar in tests/test_frontend_scale_gpu.py)."""
    c, pos, og, grads, scales = grad_case
    res, _, _, bad, _ = _statement(c, pos=pos, absolute=False, **dict(knobs))
    worst = 0.0
    for k in grads:
        g, r = bad[k].detach().reshape(-1), grads[k].detach().reshape(-1)
        ok = ~(torch.isnan(g) | torch.isnan(r))
        worst = max(worst, _worst(g[ok], r[ok], scales[k].reshape(-1)[ok]))
    print(f"[frontend ref cpu] near miss '{name}': worst err/S {worst:.3g} (bar {BAR:.3g})")
    assert worst > 4 * BAR

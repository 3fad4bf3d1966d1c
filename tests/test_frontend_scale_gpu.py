"""The frontend step at the bench shape (bench.make_host_inputs(48, 20, 1235): 48 edges over 20 keyframes, 48 x 64 x 128
fp16 maps) against the float64 statement of CorrBlock's data path in tests/frontend_ref.py: the pyramid build, three
consecutive cumulative-mask lookups, and the lookup backward in every form the bench and the training path use.  No
part of it needs the reference build.

Inputs are the bench's own, plus coordinate probes (NaN, +-inf, +-1e10, 2^31, borders) in edges 0 and 47 and Gaussian
means hanging over every border, far outside, and NaN in edges 1 and 46.  Every value of every edge is compared, a few
edges at a time; NaN patterns must be identical.

Bars: |got - ref| <= BAR S + slack per value, S = sum |terms| of the same sum (frontend_ref.py), never a global maximum.
  * BUILD_BAR = 1e-5: the volume is built on tensor cores, whose own accumulation is coarser than IEEE fp32 (the floor
    stated in test_build_gpu.py::test_build_backward_fmaps_tf32_split_matches_fp64: 1e-5 of the result's magnitude;
    S >= |value|);
  * LOOKUP_BAR = 2^-20: a looked-up value is 4 fp32 products of fp32-formed weights summed: <= 8 roundings of 2^-24 S;
    the mask (sigmoid of a 9-tap variance) to the same bar on its own scale m (1 - m) S_var + m;
  * GRAD_BAR = 2^-16: the longest fp32 sums of the backward are the Gaussian head's (81 window taps of the merged
    gradient, itself up to 4 levels): n 2^-24 S with n <= 256.  The level-0/1 gradients are accumulated in fixed point
    scaled to the pixel's largest upstream gradient (lookup_fused_bwd.cu): each contribution is rounded to 2^-23 of that
    magnitude, so those values (and the Gaussian-head gradients that read them) get that much slack per contribution.
The level-1 positions of the backward are the kernel's own (its masks are checked in the forward test); see
frontend_ref.py for why."""
import os
import sys
import time

import pytest
import torch

import frontend_ref as fr
from test_backend_scale_gpu import _probe

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E, T, SEED = 48, 20, 1235
H, W = 48, 64
P = H * W
CHUNK = 4
BUILD_BAR = 1e-5
LOOKUP_BAR = 2.0 ** -20
GRAD_BAR = 2.0 ** -16
CALLS = 3
PROBE_COORD_EDGES = (0, 47)
PROBE_MEAN_EDGES = (1, 46)


@pytest.fixture(scope="module", autouse=True)
def _report():
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    torch.cuda.synchronize()
    print(f"\n[frontend scale] module time {time.perf_counter() - t0:.1f} s, peak allocated "
          f"{torch.cuda.max_memory_allocated() / 2**30:.2f} GiB")


def _probe_means(m, e):
    """Windows over every border, far outside, and NaN, in the first row and column of edge e (m [E,H,W,2])."""
    vals = [(-3.5, 10.0), (W + 2.25, 20.0), (30.0, -2.75), (40.0, H + 3.5), (-4.5, -4.5), (W + 3.0, H + 3.0),
            (W - 0.5, H - 0.5), (1e9, 5.0), (5.0, -1e9), (float("nan"), 7.0), (9.0, float("nan")), (-100.0, 100.0)]
    for k, (x, y) in enumerate(vals):
        m[e, 0, k] = torch.tensor([x, y])
        m[e, k + 1, 0] = torch.tensor([x, y])


@pytest.fixture(scope="module")
def setup():
    sys.path.insert(0, ROOT)
    try:
        import bench
    finally:
        sys.path.remove(ROOT)
    import lgu_slam_b200
    host = bench.make_host_inputs(E, T, SEED, pin=False)
    for e in PROBE_COORD_EDGES:
        _probe(host["coords"], e, 0 if e == PROBE_COORD_EDGES[0] else P - 15)
    for e in PROBE_MEAN_EDGES:
        _probe_means(host["means"], e)
    d = {k: v.cuda() for k, v in host.items()}
    ops = lgu_slam_b200.ops
    hi, _ = ops.pack_fmaps(d["fmaps"])
    pyr = ops.build_pyramid(hi, None, d["ii"], d["jj"], H, W, means=d["means"], covs=d["covs"], den=d["den"],
                            num_levels=4, gauss_radius=4, precision=1)
    torch.cuda.synchronize()
    return dict(ops=ops, d=d, hi=hi, pyr=pyr)


def _chunks():
    return [(a, min(E, a + CHUNK)) for a in range(0, E, CHUNK)]


class Worst:
    """Per output: the worst (|got - ref| - slack)+ / S and how many values needed their slack."""

    def __init__(self):
        self.w, self.slack, self.n = {}, {}, {}

    def add(self, name, got, ref, scale, slack=None, bar=GRAD_BAR):
        got, ref = got.reshape(-1), ref.detach().reshape(-1)
        gn, rn = torch.isnan(got), torch.isnan(ref)
        assert torch.equal(gn, rn), f"{name}: NaN patterns differ at {int((gn != rn).sum())} values"
        ok = ~rn
        raw = (got[ok].double() - ref[ok]).abs()
        s = torch.nan_to_num(scale.reshape(-1)[ok], nan=0.0)
        err = raw
        used = 0
        if slack is not None:
            sl = slack.reshape(-1)[ok]
            err = (raw - sl).clamp(min=0.0)
            used = int(((raw > bar * s) & (sl > 0)).sum())
        ratio = torch.where(err == 0, torch.zeros_like(err), err / s)
        w = float(ratio.max()) if ratio.numel() else 0.0
        self.w[name] = max(self.w.get(name, 0.0), w)
        self.slack[name] = self.slack.get(name, 0) + used
        self.n[name] = self.n.get(name, 0) + int(ok.sum())
        return w

    def report(self, tag, bars):
        for k in self.w:
            print(f"[frontend scale] {tag} {k}: worst err/S {self.w[k]:.3g} (bar {bars[k]:.3g}), "
                  f"{self.slack[k]} of {self.n[k]} values needed slack")
        for k in self.w:
            assert self.w[k] <= bars[k], f"{tag} {k}: {self.w[k]:.3g} > {bars[k]:.3g}"


def _maps(d, a, b):
    f = d["fmaps"]
    return f[d["ii"][a:b].long()].double(), f[d["jj"][a:b].long()].double()


# ------------------------------------------------------------------------------------------------ a. build
@pytest.mark.parametrize("given_den", [True, False])
def test_build_matches_fp64(setup, given_den):
    s = setup
    d, ops = s["d"], s["ops"]
    pyr = s["pyr"] if given_den else ops.build_pyramid(s["hi"], None, d["ii"], d["jj"], H, W, means=d["means"],
                                                       covs=d["covs"], den=None, num_levels=4, gauss_radius=4, precision=1)
    rep = Worst()
    with torch.no_grad():
        for a, b in _chunks():
            f1, f2 = _maps(d, a, b)
            V, S_V, _ = fr.volume(f1, f2)
            den = d["den"][a:b].double() if given_den else \
                6.28 * torch.sqrt(d["covs"][a:b, ..., 0].double() * d["covs"][a:b, ..., 1].double())
            levels, scales, _ = fr.build(V, S_V, d["means"][a:b].double(), d["covs"][a:b].double(), den, H, W)
            for l in range(4):
                rep.add(f"level {l}", pyr[l][a:b], levels[l], scales[l])
            del V, S_V, levels, scales
    assert torch.isnan(pyr[0][PROBE_MEAN_EDGES[0]]).any()
    rep.report(f"build (den {'given' if given_den else 'formed'})", dict.fromkeys(rep.w, BUILD_BAR))
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ b. forward
def _forward_reference(s, a, b, knobs=None):
    """Three cumulative calls of the statement on the kernel's own pyramid: per call (corr, scale, slack, mask,
    mask scale)."""
    d, pyr = s["d"], s["pyr"]
    levels = [t[a:b].reshape(b - a, P, -1).double() for t in pyr]
    o0 = d["off0"][a:b].reshape(b - a, P, 98).double()
    o1 = d["off1"][a:b].reshape(b - a, P, 98).double()
    out = []
    for _ in range(CALLS):
        r = fr.lookup(levels, d["coords"][a:b].reshape(b - a, P, 2), o0, o1, H, W, **(knobs or {}))
        o1 = r["off1"]
        out.append((r["corr"], r["scale"], r["slack"], r["mask"], r["mask_scale"]))
    return out


def _forward_kernel(s):
    d, ops = s["d"], s["ops"]
    cum = torch.ones(E, H, W, device="cuda")
    res = []
    for _ in range(CALLS):
        corr, mask = ops.corr_lookup_fused(s["pyr"], d["coords"], d["off0"], d["off1"], 3, return_mask=True, cum_mask=cum)
        res.append((corr, mask))
    return res, cum


def test_three_cumulative_lookups_match_fp64(setup):
    s = setup
    got, _ = _forward_kernel(s)
    rep = Worst()
    nan_mask_cases = 0
    with torch.no_grad():
        for a, b in _chunks():
            ref = _forward_reference(s, a, b)
            for k, (corr, scale, slack, m, ms) in enumerate(ref):
                rep.add(f"call {k} corr", got[k][0][a:b].reshape(b - a, 196, P).transpose(1, 2), corr, scale, slack,
                        LOOKUP_BAR)
                rep.add(f"call {k} mask", got[k][1][a:b], m, ms)
            # the case a NaN mask once broke: finite coordinates, a NaN mask (a mask tap reads a NaN pyramid value) and
            # level-2 taps 0..29 -- whose offsets are zero, not masked -- reading finite, nonzero values
            c = s["d"]["coords"][a:b].reshape(b - a, P, 2)
            lvl2 = ref[0][0][..., 98:128]
            case = torch.isfinite(c).all(-1) & torch.isnan(ref[0][3]) & \
                (torch.isfinite(lvl2) & (lvl2 != 0)).any(-1)
            nan_mask_cases += int(case.sum())
    assert torch.isnan(got[0][0][PROBE_COORD_EDGES[0]]).any()
    print(f"[frontend scale] forward: {nan_mask_cases} pixels with finite coordinates, a NaN mask and finite level-2 taps")
    assert nan_mask_cases > 0
    rep.report("forward", dict.fromkeys(rep.w, LOOKUP_BAR))


# ------------------------------------------------------------------------------------------------ c. backward
def _backward_reference(s, a, b, off1_pos, knobs=None):
    """fp64 autograd of the build's Gaussian head + one lookup, on the kernel's pyramid values (straight-through: value
    from the kernel's levels, derivative from the statement's build).  Returns {name: (ref, scale, slack)}."""
    d, pyr = s["d"], s["pyr"]
    knobs = dict(knobs or {})
    bk = {k: knobs.pop(k) for k in ("level3_share",) if k in knobs}
    n = b - a
    f1, f2 = _maps(d, a, b)
    with torch.no_grad():
        V, S_V, _ = fr.volume(f1, f2)
    leaf = lambda t: t.double().requires_grad_()
    means, covs, den = leaf(d["means"][a:b]), leaf(d["covs"][a:b]), leaf(d["den"][a:b])
    means_a, covs_a, den_a = leaf(d["means"][a:b].abs()), leaf(d["covs"][a:b].abs()), leaf(d["den"][a:b].abs())
    B, _, Ba = fr.build(V, S_V, means, covs, den, H, W, None, means_a, covs_a, den_a, **bk)
    del V
    L, La = [], []
    for l in range(4):
        k = pyr[l][a:b].reshape(n, P, -1).double()
        L.append(k + (B[l] - B[l].detach()))
        La.append(k.abs() + (Ba[l] - Ba[l].detach()))
    o0, o0a = leaf(d["off0"][a:b].reshape(n, P, 98)), leaf(d["off0"][a:b].reshape(n, P, 98).abs())
    o1, o1a = leaf(d["off1"][a:b].reshape(n, P, 98)), leaf(d["off1"][a:b].reshape(n, P, 98).abs())
    g = d["corr_grad"][a:b].reshape(n, 196, P).transpose(1, 2).double()
    fxp = 2.0 ** -23 * g[..., :98].abs().amax(-1)
    r = fr.lookup(L, d["coords"][a:b].reshape(n, P, 2), o0, o1, H, W, La, o0a, o1a, off1_pos=off1_pos[a:b].reshape(n, P, 98),
                  with_slack=False, fxp=fxp, **knobs)
    names = ["gv0", "gv1", "gv2", "gv3", "off0", "off1", "means", "covs", "den"]
    ref = torch.autograd.grad((r["corr"] * g).sum(), L + [o0, o1, means, covs, den], retain_graph=True)
    sc = torch.autograd.grad((r["corr_a"] * g.abs()).sum(), La + [o0a, o1a, means_a, covs_a, den_a], retain_graph=True)
    fs = torch.autograd.grad(r["fxp"], [La[0], La[1], means_a, covs_a, den_a])
    slack = [fs[0], fs[1], None, None, None, None, fs[2], fs[3], fs[4]]
    return {k: (x.detach(), y.detach(), z) for k, x, y, z in zip(names, ref, sc, slack)}


def _compare(rep, ref, a, b, got):
    n = b - a
    for name, t in got.items():
        if t is None:
            continue
        t = t[a:b]
        t = t.reshape(n, P, -1) if name.startswith("gv") or name.startswith("off") else t
        r, sc, sl = ref[name]
        rep.add(name, t.reshape(r.shape), r, sc, sl)


MODES = ["fused", "window", "levels", "accumulate"]


def _kernel_backward(s, mode):
    """The lookup backward of one bench step (one forward from a fresh block) in the given form: the gradients and the
    fp32 post-mask offsets the kernel sampled with."""
    d, ops, pyr = s["d"], s["ops"], s["pyr"]
    gh = (d["means"], d["covs"], d["den"])
    if mode == "accumulate":                       # the training form: offset[1] updated in place, level gradients added
        off1 = d["off1"].clone()
        _, mask = ops.corr_lookup_fused(pyr, d["coords"], d["off0"], off1, 3, return_mask=True)
        bufs = [torch.zeros_like(t) for t in pyr]
        res = ops.corr_lookup_fused_backward(pyr, d["coords"], d["off0"], off1, mask, d["corr_grad"], accumulate_into=bufs)
        assert all(x is y for x, y in zip(res[:4], bufs))
        gm, gc, gd = ops.build_backward_gauss(*gh, pyr[0], list(res[:4]), 4)
        return dict(zip(["gv0", "gv1", "gv2", "gv3", "off0", "off1"], res[:6]), means=gm, covs=gc, den=gd), off1
    cum = torch.ones(E, H, W, device="cuda")
    _, mask = ops.corr_lookup_fused(pyr, d["coords"], d["off0"], d["off1"], 3, return_mask=True, cum_mask=cum)
    if mode == "fused":
        res = ops.corr_lookup_fused_backward(pyr, d["coords"], d["off0"], d["off1"], mask, d["corr_grad"], cum_mask=cum,
                                             gauss_head=gh)
        gm, gc, gd = res[6:9]
    elif mode == "window":
        res = ops.corr_lookup_fused_backward(pyr, d["coords"], d["off0"], d["off1"], mask, d["corr_grad"], cum_mask=cum,
                                             gauss_window_means=d["means"])
        gm, gc, gd = ops.build_backward_gauss(*gh, pyr[0], None, 4, window=res[6])
    else:
        res = ops.corr_lookup_fused_backward(pyr, d["coords"], d["off0"], d["off1"], mask, d["corr_grad"], cum_mask=cum)
        gm, gc, gd = ops.build_backward_gauss(*gh, pyr[0], list(res[:4]), 4)
    pos = d["off1"] * cum.unsqueeze(-1)            # offset[1] * cum_mask, the product both kernels form in fp32
    return dict(zip(["gv0", "gv1", "gv2", "gv3", "off0", "off1"], res[:6]), means=gm, covs=gc, den=gd), pos


@pytest.mark.parametrize("mode", MODES)
def test_lookup_backward_matches_fp64_autograd(setup, mode):
    s = setup
    got, pos = _kernel_backward(s, mode)
    rep = Worst()
    for a, b in _chunks():
        ref = _backward_reference(s, a, b, pos)
        _compare(rep, ref, a, b, got)
        del ref
    assert torch.isnan(got["off0"][PROBE_COORD_EDGES[0]]).any() and torch.isnan(got["means"][PROBE_MEAN_EDGES[0]]).any()
    del got
    torch.cuda.empty_cache()
    rep.report(f"backward ({mode})", dict.fromkeys(rep.w, GRAD_BAR))


# ------------------------------------------------------------------------------------------------ f. near misses
NEAR_MISSES = [
    ("biased variance", dict(biased_var=True)),
    ("no mask-path gradient into level 1", dict(drop_mask_grad=True)),
    ("per-corner gating (Q4)", dict(per_corner=True)),
    ("dx and 1 - dx swapped on level 0", dict(swap_dx_level=0)),
    ("dx and 1 - dx swapped on level 1", dict(swap_dx_level=1)),
    ("dx and 1 - dx swapped on level 3", dict(swap_dx_level=3)),
    ("level 3 weighted 1/16", dict(level3_share=1.0 / 16.0)),
]


def test_the_bars_reject_near_misses(setup):
    """Each near miss of the statement, judged against the correct statement's scales and slack on two edges of this
    input, must exceed the bars by far, in the forward (values) or the backward (gradients).  (A corr gradient that
    flows through the Gaussian branch changes only the feature-map gradients: tests/test_frontend_reference_cpu.py.)"""
    s = setup
    a, b = 2, 4
    pos = s["d"]["off1"].clone()
    with torch.no_grad():
        fwd = _forward_reference(s, a, b)
    # the statement's own post-mask offsets (one call): the near misses move positions only through the mask
    pos[a:b] = fwd[0][3].unsqueeze(-1).mul(s["d"]["off1"][a:b].reshape(b - a, P, 98).double()).float().view_as(pos[a:b])
    ref = _backward_reference(s, a, b, pos)
    for name, knobs in NEAR_MISSES:
        worst = 0.0
        fk = {k: v for k, v in knobs.items() if k != "level3_share"}
        if fk:
            with torch.no_grad():
                bad = _forward_reference(s, a, b, fk)
            for (c, sc, sl, m, ms), (c2, _, _, m2, _) in zip(fwd, bad):
                ok = ~(torch.isnan(c) | torch.isnan(c2))
                err = ((c2 - c).abs() - sl).clamp(min=0)[ok] / sc[ok]
                worst = max(worst, float(torch.nan_to_num(err, nan=0.0).max()) / LOOKUP_BAR)
        badb = _backward_reference(s, a, b, pos, knobs)
        for k, (r, sc, sl) in ref.items():
            x = badb[k][0]
            ok = ~(torch.isnan(r) | torch.isnan(x))
            err = (x - r).abs()
            if sl is not None:
                err = (err - sl).clamp(min=0)
            err = torch.where(err[ok] == 0, torch.zeros_like(err[ok]), err[ok] / sc[ok])
            worst = max(worst, float(torch.nan_to_num(err, nan=0.0).max()) / GRAD_BAR)
        print(f"[frontend scale] near miss '{name}': worst err/S {worst:.3g} x its bar")
        assert worst > 16, name
        del badb
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ d. feature-map gradients
FMAPS_BAR = 1e-5


def test_build_backward_fmaps_matches_fp64(setup):
    """build_backward_fmaps (tcgen05 kind::tf32, 3-term split) on the level gradients of the bench step's backward,
    against fp64 autograd of V = (f1/4)^T (f2/4) pooled into the 4 levels.  Bar: FMAPS_BAR = 1e-5, the tensor-core
    floor stated in test_build_gpu.py::test_build_backward_fmaps_tf32_split_matches_fp64 (the split itself is 2^-21 per
    product).  An edge whose level gradients hold a NaN (the coordinate probes) has NaN feature-map gradients wherever
    the sums reach it, which is every g_f2 value of that edge; those edges are left out and counted."""
    s = setup
    d, ops = s["d"], s["ops"]
    got, _ = _kernel_backward(s, "levels")
    grads = [got[f"gv{l}"] for l in range(4)]
    f = d["fmaps"].float()
    f1, f2 = f[d["ii"].long()].contiguous(), f[d["jj"].long()].contiguous()
    g1, g2 = ops.build_backward_fmaps(grads, f1, f2)
    bad = torch.stack([torch.isnan(g.reshape(E, -1)).any(1) for g in grads]).any(0)
    rep = Worst()
    for a, b in _chunks():
        keep = [e for e in range(a, b) if not bad[e]]
        if not keep:
            continue
        idx = torch.tensor(keep, device="cuda")
        a1, a2 = f1[idx].double().requires_grad_(), f2[idx].double().requires_grad_()
        b1, b2 = f1[idx].double().abs().requires_grad_(), f2[idx].double().abs().requires_grad_()
        V, _, Va = fr.volume(a1, a2, b1, b2)
        lv, la = [V], [Va]
        for l in range(1, 4):
            pool = lambda t: torch.nn.functional.avg_pool2d(t.reshape(-1, 1, H >> (l - 1), W >> (l - 1)), 2, 2)
            lv.append(pool(lv[-1]).reshape(len(keep), P, -1))
            la.append(pool(la[-1]).reshape(len(keep), P, -1))
        gl = [g[idx].reshape(len(keep), P, -1).double() for g in grads]
        ref = torch.autograd.grad(lv, [a1, a2], gl)
        sc = torch.autograd.grad(la, [b1, b2], [g.abs() for g in gl])
        rep.add("g_f1", g1[idx], ref[0], sc[0], bar=FMAPS_BAR)
        rep.add("g_f2", g2[idx], ref[1], sc[1], bar=FMAPS_BAR)
        del V, Va, lv, la, ref, sc
    n_bad = int(bad.sum())
    print(f"[frontend scale] build_backward_fmaps: {E - n_bad} edges compared, {n_bad} with NaN level gradients left out")
    assert n_bad <= len(PROBE_COORD_EDGES) + len(PROBE_MEAN_EDGES)
    rep.report("build_backward_fmaps", dict.fromkeys(rep.w, FMAPS_BAR))
    del got, grads, g1, g2
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ e. training chain
# Each gradient of the chain is a sum of chain-rule terms, each term a product of factors from three kinds of stage: the
# tensor-core build (<= BUILD_BAR of its scale), fp32 lookups and backward sums (<= GRAD_BAR) and the tensor-core
# feature-map products (<= FMAPS_BAR).  Relative errors of factors add, so a term is within the sum of the three bars of
# its own scale, and the absolute graph sums |terms|: the chain's bar is that sum, 3.5e-5.
TRAIN_BAR = BUILD_BAR + GRAD_BAR + FMAPS_BAR
TRAIN_CHUNK = 4
LEAVES = ("f1", "f2", "mean", "cov", "det", "off0", "off1")


def _train_case(n, seed):
    """fp32 maps (the hi/lo precision-2 build), the bench's Gaussian head and offsets for n edges, three coordinate sets
    (probes without NaN: a NaN coordinate makes every g_f2 value of its edge NaN) and three upstream gradients."""
    sys.path.insert(0, ROOT)
    try:
        import bench
    finally:
        sys.path.remove(ROOT)
    import inputs
    host = bench.make_host_inputs(n, T, seed, pin=False)
    _probe_means(host["means"], 1)
    host["means"] = torch.nan_to_num(host["means"], nan=-50.0)     # a NaN mean likewise: windows over borders only
    g = inputs.gen(seed + 11)
    c0 = host["coords"].clone()
    _probe(c0, 0, 0)
    coords = [torch.nan_to_num(c0, nan=-1e10)] + [c0.nan_to_num(nan=-1e10) + 0.75 * torch.randn(c0.shape, generator=g)
                                                  for _ in range(CALLS - 1)]
    cv = host["covs"]
    case = dict(f1=torch.randn(n, 128, H, W, generator=g), f2=torch.randn(n, 128, H, W, generator=g),
                mean=host["means"], cov=cv, det=(cv[..., 0] * cv[..., 1]).reshape(n, P),
                off0=host["off0"], off1=host["off1"])
    case = {k: v.contiguous().cuda() for k, v in case.items()}
    case["coords"] = [c.contiguous().cuda() for c in coords]
    case["wts"] = [host["corr_grad"].cuda()] + [torch.randn(n, 196, H, W, generator=g).cuda() for _ in range(CALLS - 1)]
    return case


def _train_kernel(case, accumulate):
    """FusedBuild + 3 x FusedCorrLookup + one backward: leaf gradients and each call's fp32 post-mask offsets."""
    from importlib import import_module
    corr = import_module("lgu-slam_b200.corr")
    lv = {k: case[k].clone().requires_grad_() for k in LEAVES}
    acc = corr.LevelGradAccumulator() if accumulate else None
    *pyr, token = corr.FusedBuild.apply(lv["f1"], lv["f2"], lv["mean"], lv["cov"], lv["det"], False, acc)
    if acc is not None:
        acc.levels = tuple(pyr)
    o1, pos, loss = lv["off1"], [], 0.0
    for k in range(CALLS):
        extra = (token, acc) if accumulate else ()
        out, o1, _ = corr.FusedCorrLookup.apply(pyr[0], pyr[1], pyr[2], pyr[3], case["coords"][k], lv["off0"], o1, *extra)
        pos.append(o1.detach().clone())
        loss = loss + (out * case["wts"][k]).sum()
    loss.backward()
    return {k: lv[k].grad for k in LEAVES}, pos


def _train_reference(case, a, b, pos, **knobs):
    """fp64 autograd of volume -> build -> 3 x lookup for edges a..b: {leaf: (ref, scale, slack)}.  Level-1 positions
    are the kernel's (pos); the fixed-point slack of the level-0/1 gradients is carried back to every leaf."""
    n = b - a
    lv = {k: case[k][a:b].double().requires_grad_() for k in LEAVES}
    la = {k: case[k][a:b].double().abs().requires_grad_() for k in LEAVES}
    bk = {k: knobs.pop(k) for k in ("corr_through_gauss", "level3_share") if k in knobs}
    V, S_V, Va = fr.volume(lv["f1"], lv["f2"], la["f1"], la["f2"])
    den, den_a = fr._elementwise(lambda t: 6.28 * torch.sqrt(t), (lv["det"],), (la["det"],))
    levels, _, levels_a = fr.build(V, S_V, lv["mean"], lv["cov"], den.view(n, H, W), H, W, Va, la["mean"], la["cov"],
                                   den_a.view(n, H, W), **bk)
    del V, Va
    o0, o0a = lv["off0"].view(n, P, 98), la["off0"].view(n, P, 98)
    o1, o1a = lv["off1"].view(n, P, 98), la["off1"].view(n, P, 98)
    loss = loss_a = fx = 0.0
    for k in range(CALLS):
        w = case["wts"][k][a:b].reshape(n, 196, P).transpose(1, 2).double()
        r = fr.lookup(levels, case["coords"][k][a:b].reshape(n, P, 2), o0, o1, H, W, levels_a, o0a, o1a,
                      off1_pos=pos[k][a:b].reshape(n, P, 98), with_slack=False,
                      fxp=2.0 ** -23 * w[..., :98].abs().amax(-1), **knobs)
        o1, o1a = r["off1"], r["off1_a"]
        loss = loss + (r["corr"] * w).sum()
        loss_a = loss_a + (r["corr_a"] * w.abs()).sum()
        fx = fx + r["fxp"]
    ref = torch.autograd.grad(loss, [lv[k] for k in LEAVES], retain_graph=True)
    sc = torch.autograd.grad(loss_a, [la[k] for k in LEAVES], retain_graph=True)
    sl = torch.autograd.grad(fx, [la[k] for k in LEAVES], allow_unused=True)
    return {k: (r_.detach(), s_.detach(), None if z is None else z.detach()) for k, r_, s_, z in zip(LEAVES, ref, sc, sl)}


@pytest.mark.parametrize("n", [48, 96])
@pytest.mark.parametrize("accumulate", [False, True])
def test_training_chain_matches_fp64_autograd(n, accumulate):
    """FusedBuild.apply + FusedCorrLookup.apply over three lookups (the later calls' offsets depend on the earlier masks,
    Q7, so the backward carries an upstream gradient on offset[1]_out), one backward, level gradients returned densely or
    accumulated in persistent buffers: every leaf gradient against fp64 autograd of the whole statement, at the bench's
    E = 48 and the training shape b n = 96.  Bar: TRAIN_BAR (above)."""
    case = _train_case(n, 2000 + n)
    got, pos = _train_kernel(case, accumulate)
    torch.cuda.synchronize()
    rep = Worst()
    for a in range(0, n, TRAIN_CHUNK):
        b = min(n, a + TRAIN_CHUNK)
        ref = _train_reference(case, a, b, pos)
        for k in LEAVES:
            r, sc, sl = ref[k]
            rep.add(k, got[k][a:b].reshape(r.shape), r, sc, sl, bar=TRAIN_BAR)
        del ref
    del got, pos
    torch.cuda.empty_cache()
    rep.report(f"training chain (E {n}, {'accumulate' if accumulate else 'dense'})", dict.fromkeys(rep.w, TRAIN_BAR))


def test_training_chain_bar_rejects_near_misses():
    """At this shape, with the kernel's positions: the corr gradient through the Gaussian branch (visible only in the
    feature-map gradients), the mask path's share of level 1 and level 3 weighted 1/16 must exceed TRAIN_BAR by a margin
    (4x).  The mask path reaches these leaves only diluted by the other level-1 terms (~6x); where its level gradient is
    compared directly (test_the_bars_reject_near_misses) the same near miss exceeds GRAD_BAR by ~10^4."""
    case = _train_case(48, 2048)
    _, pos = _train_kernel(case, False)
    a, b = 4, 6
    ref = _train_reference(case, a, b, pos)
    for name, knobs in (("corr gradient through the Gaussian branch", dict(corr_through_gauss=True)),
                        ("no mask-path gradient into level 1", dict(drop_mask_grad=True)),
                        ("level 3 weighted 1/16", dict(level3_share=1.0 / 16.0))):
        bad = _train_reference(case, a, b, pos, **knobs)
        worst = 0.0
        for k in LEAVES:
            r, sc, sl = ref[k]
            x = bad[k][0]
            ok = ~(torch.isnan(r) | torch.isnan(x))
            err = (x - r).abs()
            if sl is not None:
                err = (err - sl).clamp(min=0)
            err = torch.where(err[ok] == 0, torch.zeros_like(err[ok]), err[ok] / sc[ok])
            worst = max(worst, float(torch.nan_to_num(err, nan=0.0).max()) / TRAIN_BAR)
        print(f"[frontend scale] training near miss '{name}': worst err/S {worst:.3g} x its bar")
        assert worst > 4, name


def test_corrblock_glue_feeds_the_checked_ops():
    """CorrBlock(fused=True) at E = 2 (GaussianMask.params -> mean / cov / det, the offset heads, FusedBuild, three
    FusedCorrLookup calls with the level-gradient accumulator): its gradients of the maps and of every learned parameter
    equal autograd of the same glue run on its own with the two fused ops' gradients -- the ops the test above checks
    against fp64 -- fed in where the glue meets them.  Identical fp32 arithmetic on both sides: 2^-20 of the sum of
    both magnitudes (reduction-order differences of cuDNN / cuBLAS only)."""
    import torch.nn as nn
    from importlib import import_module
    corr = import_module("lgu-slam_b200.corr")
    import inputs
    g = inputs.gen(77)
    n = 2
    torch.manual_seed(78)
    ofsMap = nn.Conv2d(256, 98, 3, padding=1).cuda()
    ofs_res = nn.Conv2d(256, 98, 3, padding=1).cuda()
    GA = corr.GaussianMask(H, W).cuda()
    with torch.no_grad():
        GA.meanMap.weight.normal_(0, 0.3)
        GA.meanMap.bias.normal_(0, 0.3)
    fm1 = torch.randn(1, n, 128, H, W, generator=g).cuda()
    fm2 = torch.randn(1, n, 128, H, W, generator=g).cuda()
    coords = [inputs.make_coords(n, H, W, H, W, g).permute(0, 2, 3, 1).contiguous().view(1, n, H, W, 2).cuda()
              for _ in range(CALLS)]
    wts = [torch.randn(1, n, 196, H, W, generator=g).cuda() for _ in range(CALLS)]
    params = [("ofsMap.weight", ofsMap.weight), ("ofsMap.bias", ofsMap.bias), ("ofs_residual.weight", ofs_res.weight),
              ("GA.map.weight", GA.map.weight), ("GA.covMap.weight", GA.covMap.weight),
              ("GA.meanMap.weight", GA.meanMap.weight), ("GA.meanMap.bias", GA.meanMap.bias)]

    def run(block):
        for _, p in params:
            p.grad = None
        f1, f2 = fm1.clone().requires_grad_(), fm2.clone().requires_grad_()
        loss = block(f1, f2)
        loss.backward()
        return [("fmap1", f1.grad), ("fmap2", f2.grad)] + [(k, p.grad.clone()) for k, p in params]

    def whole(f1, f2):
        blk = corr.CorrBlock(ofsMap, ofs_res, GA, f1, f2, fused=True)
        assert blk._gacc is not None
        loss = 0.0
        for c, w in zip(coords, wts):
            out, mean_n, theta = blk(c)
            loss = loss + (out * w).sum() + (mean_n.square().sum() + theta.sum()) * 1e-2
        return loss

    def glued(f1, f2):
        # the glue by hand: the same modules, then the two fused ops as the checked test calls them
        E_ = n
        t = torch.cat((f1.reshape(E_, 128, H, W), f2.reshape(E_, 128, H, W)), dim=1)
        off = corr._generate_offsets(ofsMap, ofs_res, t.float(), True)
        mean, cov, det = GA.params(t.permute(0, 2, 3, 1).contiguous().float())
        acc = corr.LevelGradAccumulator()
        *pyr, token = corr.FusedBuild.apply(f1.reshape(E_, 128, H, W), f2.reshape(E_, 128, H, W), mean, cov, det, False, acc)
        acc.levels = tuple(pyr)
        o1, loss = off[1], 0.0
        for c, w in zip(coords, wts):
            out, o1, _ = corr.FusedCorrLookup.apply(pyr[0], pyr[1], pyr[2], pyr[3], c.reshape(E_, H, W, 2).contiguous(),
                                                    off[0], o1, token, acc)
            loss = loss + (out.view(1, E_, 196, H, W) * w).sum() + \
                (mean.view(1, E_, H, W, 2).square().sum() + (2 * det).sum()) * 1e-2
        return loss

    prev = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        a, b = run(whole), run(glued)
    finally:
        torch.backends.cudnn.deterministic = prev
    worst = 0.0
    for (k, x), (_, y) in zip(a, b):
        assert x is not None and torch.isfinite(x).all() and (x != 0).any(), k
        err = (x - y).abs() / (x.abs() + y.abs()).clamp(min=1e-30)
        worst = max(worst, float(err.max()))
        assert float(err.max()) <= 2.0 ** -20, f"{k}: {float(err.max()):.3g}"
    print(f"[frontend scale] CorrBlock(fused=True) glue: worst |a - b| / (|a| + |b|) {worst:.3g} over "
          f"{len(a)} gradients")

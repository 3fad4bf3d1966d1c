"""GPU parity of the fused 4-level lookup (lgu_corr_lookup_fused, one TMA-staged launch) against the oracle's
composition of the reference ops (CorrBlock.__call__, corr.py:88-109): r=1 mask lookup on level 1 -> var -> sigmoid
-> offset[1] *= mask -> four deformable r=3 lookups -> cat.

Bars: levels 0, 2, 3 (their offsets do not depend on the mask) bit-exact, including the zero pattern of gated
taps; level 1 within 1e-5 abs (its offsets are scaled by sigmoid(var), whose fp32 rounding differs between
torch's Welford reduction and the kernel's two-pass variance by a few ulp); the in-place side effects on the
offsets (Q5 centre-tap zeroing, Q7 cumulative mask) match within 1e-6."""
import pytest
import torch

import inputs

pytestmark = pytest.mark.gpu
ATOL = 1e-5


def _case(E, seed, big_offsets=False, probes=False):
    c = inputs.frontend_case(E=E, T=max(3, E // 2), seed=seed, half_fmaps=True)
    if big_offsets:   # offsets beyond the staged box (|o| >= 4): exercises the direct-global slow path
        g = inputs.gen(seed + 1)
        c["offsets"][0] = (9.0 * torch.randn(E, 48, 64, 98, generator=g)).contiguous()
        c["offsets"][1] = (7.0 * torch.randn(E, 48, 64, 98, generator=g)).contiguous()
    if probes:
        co = c["coords"]
        co[0, 0, 0] = torch.tensor([float("nan"), 3.0])
        co[0, 0, 1] = torch.tensor([float("inf"), -float("inf")])
        co[0, 0, 2] = torch.tensor([1e30, -1e30])
        co[0, 0, 3] = torch.tensor([-0.0, 47.0])
        co[0, 0, 4] = torch.tensor([63.0, 47.999])
        co[0, 0, 5] = torch.tensor([-1.0, -1.0])
        co[0, 0, 6] = torch.tensor([2147483648.0, 5.0])
    return c


def _pyramid(oracle, c):
    f1 = c["fmaps"][c["ii"].long()].contiguous()
    f2 = c["fmaps"][c["jj"].long()].contiguous()
    return oracle.build_pyramid(f1, f2, c["means"], c["covs"], 4, 4, False)


@pytest.mark.parametrize("E,seed,big,probes", [(2, 51, False, False), (3, 52, False, True), (2, 53, True, True)])
def test_fused_lookup_matches_oracle_composition(ops, oracle, E, seed, big, probes):
    c = _case(E, seed, big, probes)
    pyr = _pyramid(oracle, c)
    offs = [o.clone() for o in c["offsets"]]
    want = oracle.corr_block_lookup(pyr, c["coords"], offs, 3)          # mutates offs like the reference
    dev = "cuda"
    off0, off1 = c["offsets"][0].to(dev), c["offsets"][1].to(dev)
    got, mask = ops.corr_lookup_fused([p.to(dev) for p in pyr], c["coords"].to(dev), off0, off1, 3, return_mask=True)
    got = got.cpu()
    assert torch.equal(torch.isnan(got), torch.isnan(want))
    for l in (0, 2, 3):
        a, b = got[:, 49 * l:49 * (l + 1)], want[:, 49 * l:49 * (l + 1)]
        assert torch.equal(torch.nan_to_num(a), torch.nan_to_num(b)), f"level {l} must be bit-exact"
    a, b = got[:, 49:98], want[:, 49:98]
    err = (torch.nan_to_num(a) - torch.nan_to_num(b)).abs().max().item()
    assert err <= ATOL, f"level 1: max abs err {err}"
    # side effects: off0 untouched; off1 <- off1 * mask for every tap (the centre tap is only READ as zero: inside
    # CorrBlock the reference zeroes a temporary copy, so the stored value survives there too)
    assert torch.equal(off0.cpu(), c["offsets"][0])
    o1 = off1.cpu().view(E, 48, 64, 49, 2)
    w1 = offs[1].view(E, 48, 64, 49, 2)
    keep = [t for t in range(49) if t != 24]
    assert torch.equal(torch.isnan(o1[..., keep, :]), torch.isnan(w1[..., keep, :]))
    assert (torch.nan_to_num(o1[..., keep, :]) - torch.nan_to_num(w1[..., keep, :])).abs().max().item() <= 1e-5
    centre = c["offsets"][1].view(E, 48, 64, 49, 2)[..., 24, :] * mask.cpu()[..., None]
    assert torch.allclose(torch.nan_to_num(o1[..., 24, :]), torch.nan_to_num(centre), atol=1e-6)
    assert mask.shape == (E, 48, 64)


def test_fused_lookup_is_cumulative_like_the_reference(ops, oracle):
    """Two consecutive calls: offset[1] is re-multiplied by each call's mask (quirk Q7)."""
    c = _case(2, 54)
    pyr = _pyramid(oracle, c)
    offs = [o.clone() for o in c["offsets"]]
    g = inputs.gen(99)
    coords2 = (c["coords"] + 0.7 * torch.randn(c["coords"].shape, generator=g)).contiguous()
    oracle.corr_block_lookup(pyr, c["coords"], offs, 3)
    want2 = oracle.corr_block_lookup(pyr, coords2, offs, 3)
    dev = "cuda"
    off0, off1 = c["offsets"][0].to(dev), c["offsets"][1].to(dev)
    pg = [p.to(dev) for p in pyr]
    ops.corr_lookup_fused(pg, c["coords"].to(dev), off0, off1, 3)
    got2 = ops.corr_lookup_fused(pg, coords2.to(dev), off0, off1, 3).cpu()
    assert (got2 - want2).abs().max().item() <= ATOL


def test_fused_lookup_equals_per_level_operators(ops):
    """Against the product's own drop-in operators at the full frontend size (E=48): identical results."""
    E = 48
    c = inputs.frontend_case(E=E, T=20, seed=55, half_fmaps=True)
    dev = "cuda"
    hi, _ = ops.pack_fmaps(c["fmaps"].half().to(dev))
    den = (6.28 * torch.sqrt(c["covs"][..., 0] * c["covs"][..., 1])).to(dev).contiguous()
    pyr = ops.build_pyramid(hi, None, c["ii"].to(dev), c["jj"].to(dev), 48, 64, means=c["means"].to(dev),
                            covs=c["covs"].to(dev), den=den)
    coords = c["coords"].to(dev)
    off0, off1 = c["offsets"][0].to(dev), c["offsets"][1].to(dev)
    got, mask = ops.corr_lookup_fused(pyr, coords, off0.clone(), off1.clone(), 3, return_mask=True)
    cc = coords.permute(0, 3, 1, 2).contiguous()
    m, = ops.corr_index_forward(pyr[1], (cc / 2).contiguous(), 1)
    mk = torch.sigmoid(torch.var(m.permute(0, 3, 4, 1, 2), dim=[3, 4]))
    assert (mk - mask).abs().max().item() <= 1e-6
    offs = [off0.clone(), off1 * mask.view(E, 48, 64, 1), torch.zeros_like(off0), torch.zeros_like(off0)]
    for l in range(4):
        want, = ops.defCorr_index_forward(pyr[l], (cc / 2 ** l).contiguous(), offs[l].view(E, 48, 64, 7, 7, 2), 3)
        assert torch.equal(got[:, 49 * l:49 * (l + 1)], want.view(E, 49, 48, 64)), f"level {l}"


def test_fused_lookup_unsupported_configuration_is_reported(ops):
    dev = "cuda"
    pyr = [torch.zeros(1, 8, 16, 8 >> l, 16 >> l, device=dev) for l in range(4)]
    with pytest.raises(RuntimeError, match="W%32"):
        ops.corr_lookup_fused(pyr, torch.zeros(1, 8, 16, 2, device=dev), torch.zeros(1, 8, 16, 98, device=dev),
                              torch.zeros(1, 8, 16, 98, device=dev), 3)


def _per_op_autograd(corr_mod, pyr, coords, off0, off1):
    """The reference's autograd graph for CorrBlock.__call__ (corr.py:88-109) on the per-level operators."""
    E = coords.shape[0]
    c = coords.permute(0, 3, 1, 2).contiguous()
    m = corr_mod.CorrSampler.apply(pyr[1], c / 2, 1)
    mask = torch.sigmoid(torch.var(m.permute(0, 3, 4, 1, 2), dim=[3, 4])).view(E, 48, 64, 1)
    off1_out = off1 * mask
    z = torch.zeros_like(off0)
    outs = []
    for l, o in enumerate((off0, off1_out, z, z.clone())):
        # like the reference inside CorrBlock, hand the sampler a COPY (`.contiguous()` of a permuted view)
        outs.append(corr_mod.DefCorrSampler.apply(pyr[l], c / 2 ** l, o.clone().view(E, 48, 64, 7, 7, 2), 3)
                    .view(E, 49, 48, 64))
    return torch.cat(outs, dim=1), off1_out


@pytest.mark.parametrize("big,probes", [(False, False), (True, False), (False, True)])
def test_fused_backward_matches_per_op_autograd(ops, big, probes):
    from importlib import import_module
    corr_mod = import_module("lgu-slam_b200.corr")
    E = 2
    c = _case(E, 61, big_offsets=big, probes=probes)
    dev = "cuda"
    g = inputs.gen(62)
    pyr_a = [torch.randn(E, 48, 64, 48 >> l, 64 >> l, generator=g).to(dev).requires_grad_() for l in range(4)]
    pyr_b = [p.detach().clone().requires_grad_() for p in pyr_a]
    coords = c["coords"].to(dev)
    off0_a, off1_a = c["offsets"][0].to(dev).requires_grad_(), c["offsets"][1].to(dev).requires_grad_()
    off0_b, off1_b = off0_a.detach().clone().requires_grad_(), off1_a.detach().clone().requires_grad_()
    g_corr = torch.randn(E, 196, 48, 64, generator=g).to(dev)
    g_off1 = (0.1 * torch.randn(E, 48, 64, 98, generator=g)).to(dev)

    out_a, off1_out_a, _ = corr_mod.FusedCorrLookup.apply(*pyr_a, coords, off0_a, off1_a)
    ((torch.nan_to_num(out_a) * g_corr).sum() + (torch.nan_to_num(off1_out_a) * g_off1).sum()).backward()
    out_b, off1_out_b = _per_op_autograd(corr_mod, pyr_b, coords, off0_b, off1_b)
    ((torch.nan_to_num(out_b) * g_corr).sum() + (torch.nan_to_num(off1_out_b) * g_off1).sum()).backward()

    def diff(x, y, what):
        # NaN / inf coordinates make the same taps NaN in both graphs: identical NaN pattern, finite values compared
        assert torch.equal(torch.isnan(x), torch.isnan(y)), f"{what}: NaN patterns differ"
        return (torch.nan_to_num(x) - torch.nan_to_num(y)).abs().max().item()

    assert diff(out_a, out_b, "corr") <= ATOL
    for l in range(4):
        err = diff(pyr_a[l].grad, pyr_b[l].grad, f"level {l} volume grad")
        scale = torch.nan_to_num(pyr_b[l].grad).abs().max().item()
        assert err <= 1e-5 * max(1.0, scale), f"level {l} volume grad: {err} (scale {scale})"
    for name, x, y in (("off0", off0_a, off0_b), ("off1", off1_a, off1_b)):
        err = diff(x.grad, y.grad, f"{name} grad")
        scale = torch.nan_to_num(y.grad).abs().max().item()
        assert err <= 1e-5 * max(1.0, scale), f"{name} grad: {err} (scale {scale})"


@pytest.mark.parametrize("H,W", [(40, 96), (8, 32), (16, 128)])
def test_fused_lookup_and_backward_on_other_grid_sizes(ops, H, W):
    """The fused kernels are generic in the grid (W % 32 == 0, H % 8 == 0): non-power-of-two level widths take the
    generic slice-streaming loop; compare against the per-level operators / their autograd graph on the GPU."""
    from importlib import import_module
    corr_mod = import_module("lgu-slam_b200.corr")
    E, dev = 2, "cuda"
    g = inputs.gen(70 + H)
    pyr = [torch.randn(E, H, W, H >> l, W >> l, generator=g).to(dev) for l in range(4)]
    coords = inputs.make_coords(E, H, W, H, W, g).permute(0, 2, 3, 1).contiguous().to(dev)
    off0 = (4 * torch.tanh(torch.randn(E, H, W, 98, generator=g))).to(dev)
    off1 = (4 * torch.tanh(torch.randn(E, H, W, 98, generator=g))).to(dev)
    # forward vs per-level operators
    o1 = off1.clone()
    got, mask = ops.corr_lookup_fused(pyr, coords, off0, o1, 3, return_mask=True)
    cc = coords.permute(0, 3, 1, 2).contiguous()
    m, = ops.corr_index_forward(pyr[1], (cc / 2).contiguous(), 1)
    mk = torch.sigmoid(torch.var(m.permute(0, 3, 4, 1, 2), dim=[3, 4]))
    assert (mk - mask).abs().max().item() <= 1e-6
    offs = [off0.clone(), off1 * mask.view(E, H, W, 1), torch.zeros_like(off0), torch.zeros_like(off0)]
    for l in range(4):
        want, = ops.defCorr_index_forward(pyr[l], (cc / 2 ** l).contiguous(), offs[l].view(E, H, W, 7, 7, 2), 3)
        assert torch.equal(got[:, 49 * l:49 * (l + 1)], want.view(E, 49, H, W)), f"level {l}"
    # backward vs the per-op autograd graph
    pa = [p.clone().requires_grad_() for p in pyr]
    pb = [p.clone().requires_grad_() for p in pyr]
    a0, a1 = off0.clone().requires_grad_(), off1.clone().requires_grad_()
    b0, b1 = off0.clone().requires_grad_(), off1.clone().requires_grad_()
    gc = torch.randn(E, 196, H, W, generator=g).to(dev)
    out_a, o1a, _ = corr_mod.FusedCorrLookup.apply(*pa, coords, a0, a1)
    (out_a * gc).sum().backward()
    c = coords.permute(0, 3, 1, 2).contiguous()
    mm = corr_mod.CorrSampler.apply(pb[1], c / 2, 1)
    msk = torch.sigmoid(torch.var(mm.permute(0, 3, 4, 1, 2), dim=[3, 4])).view(E, H, W, 1)
    z = torch.zeros_like(off0)
    outs = [corr_mod.DefCorrSampler.apply(pb[l], c / 2 ** l, o.clone().view(E, H, W, 7, 7, 2), 3).view(E, 49, H, W)
            for l, o in enumerate((b0, b1 * msk, z, z.clone()))]
    (torch.cat(outs, 1) * gc).sum().backward()
    for l in range(4):
        scale = max(1.0, pb[l].grad.abs().max().item())
        assert (pa[l].grad - pb[l].grad).abs().max().item() <= 1e-5 * scale, f"level {l} volume grad"
    for a, b in ((a0, b0), (a1, b1)):
        assert (a.grad - b.grad).abs().max().item() <= 1e-5 * max(1.0, b.grad.abs().max().item())


@pytest.mark.parametrize("big", [False, True])
def test_fused_backward_accumulate_equals_sum_of_dense_calls(ops, big):
    """Training clip (droid_net.py:187-222): three lookups of one pyramid.  The accumulate entry point adds each call's
    footprints into persistent buffers (16-byte L2 reductions); the dense entry point returns one dense gradient per
    call.  The sequential fp32 sum of the dense results is what the accumulators must hold (fp32 add of the same
    terms in the same order; the reductions flush denormals, hence the 1e-30 allowance), and the offset gradients
    of every call must be bit-identical."""
    E, dev = 2, "cuda"
    g = inputs.gen(71)
    pyr = [torch.randn(E, 48, 64, 48 >> l, 64 >> l, generator=g).to(dev) for l in range(4)]
    acc = [torch.zeros_like(p) for p in pyr]
    want = [torch.zeros_like(p) for p in pyr]
    for step in range(3):
        c = _case(E, 72 + step, big_offsets=big, probes=(step == 1))     # NaN / inf / 2^31 coordinates in one call
        coords, off0, off1 = c["coords"].to(dev), c["offsets"][0].to(dev), c["offsets"][1].to(dev)
        _, mask = ops.corr_lookup_fused(pyr, coords, off0, off1, 3, return_mask=True)
        g_corr = torch.randn(E, 196, 48, 64, generator=g).to(dev)
        g_up = (0.1 * torch.randn(E, 48, 64, 98, generator=g)).to(dev)
        dense = ops.corr_lookup_fused_backward(pyr, coords, off0, off1, mask, g_corr, g_up)
        got = ops.corr_lookup_fused_backward(pyr, coords, off0, off1, mask, g_corr, g_up, accumulate_into=acc)
        for l in range(4):
            assert got[l] is acc[l]
            want[l] += dense[l]
        assert torch.equal(torch.nan_to_num(got[4]), torch.nan_to_num(dense[4])) and \
            torch.equal(torch.nan_to_num(got[5]), torch.nan_to_num(dense[5])), "offset gradients differ"
    for l in range(4):
        assert torch.equal(torch.isnan(acc[l]), torch.isnan(want[l])), f"level {l}: NaN patterns differ"
        err = (torch.nan_to_num(acc[l]) - torch.nan_to_num(want[l])).abs().max().item()
        # out-of-box taps (|offset| >= 4, `big`) go through scalar atomics whose order is not fixed
        tol = 1e-30 if not big else 1e-5 * max(1.0, torch.nan_to_num(want[l]).abs().max().item())
        assert err <= tol, f"level {l}: accumulated gradient differs from the sum of dense calls by {err}"


def test_fused_lookup_cumulative_mask_mode_equals_write_back_mode(ops):
    """lgu_corr_lookup_fused_cum keeps offset[1] pristine and the running product of the masks in a [E,H,W] buffer;
    three consecutive calls must give what the write-back entry point gives (the reference's cumulative
    `self.offset[1] *= mask`, Q7): levels 0, 2, 3 bit-identical, level 1 within 1e-5 of the largest value (o*(m1*m2) vs
    (o*m1)*m2 moves an offset by <= 2 ulp, times the local slope of a white-noise pyramid with |V| up to ~5), and
    off1 * cum_mask equal to the written-back offsets within 2 ulp of the offset magnitude."""
    E, dev = 2, "cuda"
    g = inputs.gen(81)
    pyr = [torch.randn(E, 48, 64, 48 >> l, 64 >> l, generator=g).to(dev) for l in range(4)]
    c = _case(E, 82)
    off0, off1 = c["offsets"][0].to(dev), c["offsets"][1].to(dev)
    wb = off1.clone()
    cum = torch.ones(E, 48, 64, device=dev)
    for step in range(3):
        coords = (c["coords"] + 0.6 * step * torch.randn(c["coords"].shape, generator=g)).contiguous().to(dev)
        want, m_w = ops.corr_lookup_fused(pyr, coords, off0, wb, 3, return_mask=True)
        keep = off1.clone()
        got, m_c = ops.corr_lookup_fused(pyr, coords, off0, off1, 3, return_mask=True, cum_mask=cum)
        assert torch.equal(off1, keep), "cum mode must not touch offset[1]"
        for l in (0, 2, 3):
            assert torch.equal(got[:, 49 * l:49 * (l + 1)], want[:, 49 * l:49 * (l + 1)]), f"call {step} level {l}"
        scale = max(1.0, want[:, 49:98].abs().max().item())
        assert (got[:, 49:98] - want[:, 49:98]).abs().max().item() <= 1e-5 * scale, f"call {step} level 1"
        assert (m_c - m_w).abs().max().item() <= 1e-6
        assert ((off1 * cum.view(E, 48, 64, 1)) - wb).abs().max().item() <= 1e-6


@pytest.mark.parametrize("accumulate", [False, True])
def test_fused_backward_cumulative_mask_form_equals_materialised_form(ops, accumulate):
    """lgu_corr_lookup_fused_backward_cum (pristine offset[1] + the running mask product) against the entry point that
    reads the materialised post-mask offsets: bit-identical level and offset gradients."""
    E, dev = 2, "cuda"
    g = inputs.gen(91)
    pyr = [torch.randn(E, 48, 64, 48 >> l, 64 >> l, generator=g).to(dev) for l in range(4)]
    c = _case(E, 92)
    coords, off0, off1 = c["coords"].to(dev), c["offsets"][0].to(dev), c["offsets"][1].to(dev)
    cum = torch.ones(E, 48, 64, device=dev)
    for _ in range(2):                                            # second call: cum_mask = m1 * m2
        _, mask = ops.corr_lookup_fused(pyr, coords, off0, off1, 3, return_mask=True, cum_mask=cum)
    g_corr = torch.randn(E, 196, 48, 64, generator=g).to(dev)
    off1_out = (off1 * cum.unsqueeze(-1)).contiguous()
    acc_a = [torch.zeros_like(p) for p in pyr] if accumulate else None
    acc_b = [torch.zeros_like(p) for p in pyr] if accumulate else None
    want = ops.corr_lookup_fused_backward(pyr, coords, off0, off1_out, mask, g_corr, accumulate_into=acc_a)
    got = ops.corr_lookup_fused_backward(pyr, coords, off0, off1, mask, g_corr, accumulate_into=acc_b, cum_mask=cum)
    for k, (a, b) in enumerate(zip(got, want)):
        assert torch.equal(a, b), f"output {k}"


@pytest.mark.parametrize("big,edge_means", [(False, False), (True, False), (False, True)])
def test_fused_backward_window_record_equals_merged_level_gradients(ops, big, edge_means):
    """lgu_corr_lookup_fused_backward_win: the 9 x 9 window record of g0 + g1/4 + g2/16 + g3/64 around floor(means) is,
    bit for bit, what avg_pool2d^T (corr.py:83-86) of the dense level gradients gives at those taps (zeros outside the
    grid), the dense gradients themselves are unchanged, and the Gaussian-head gradients from the record equal the ones
    from the four level gradients (gaussianMask_cuda.py:77-86 backward).  `big`: offsets beyond the staged boxes, whose
    contributions travel by global atomics and are not in the shared-memory boxes the record is normally formed from."""
    E, dev, H, W = 2, "cuda", 48, 64
    g = inputs.gen(131)
    pyr = [torch.randn(E, H, W, H >> l, W >> l, generator=g).to(dev) for l in range(4)]
    c = _case(E, 132, big_offsets=big)
    coords, off0, off1 = c["coords"].to(dev), c["offsets"][0].to(dev), c["offsets"][1].to(dev)
    means, covs = c["means"].to(dev).contiguous(), c["covs"].to(dev).contiguous()
    if edge_means:                                                # windows hanging over every border, far outside, NaN
        means[0, 0, 0] = torch.tensor([-3.5, -2.25]); means[0, 0, 1] = torch.tensor([66.0, 49.5])
        means[0, 0, 2] = torch.tensor([-100.0, 1e9]); means[0, 0, 3] = torch.tensor([float("nan"), 5.0])
        means[0, 0, 4] = torch.tensor([63.9, 47.9]); means[0, 0, 5] = torch.tensor([0.0, 0.0])
    den = (6.28 * torch.sqrt(covs[..., 0] * covs[..., 1])).contiguous()
    cum = torch.ones(E, H, W, device=dev)
    _, mask = ops.corr_lookup_fused(pyr, coords, off0, off1, 3, return_mask=True, cum_mask=cum)
    g_corr = torch.randn(E, 196, H, W, generator=g).to(dev)
    want = ops.corr_lookup_fused_backward(pyr, coords, off0, off1, mask, g_corr, cum_mask=cum)
    got = ops.corr_lookup_fused_backward(pyr, coords, off0, off1, mask, g_corr, cum_mask=cum, gauss_window_means=means)
    assert len(got) == 7
    for k in (4, 5):
        assert torch.equal(got[k], want[k]), f"output {k}"
    for k in range(4):                                            # out-of-box taps arrive by float atomics: order-dependent
        if big:
            assert (got[k] - want[k]).abs().max().item() <= 1e-5 * max(1.0, want[k].abs().max().item())
        else:
            assert torch.equal(got[k], want[k]), f"output {k}"
    # the record, from the dense gradients of the SAME call
    gl = got[:4]
    merged = gl[0].clone()
    for l, f in ((1, 0.25), (2, 0.0625), (3, 0.015625)):
        up = gl[l].repeat_interleave(1 << l, dim=3).repeat_interleave(1 << l, dim=4)
        merged = merged + up * f                                  # same order of fp32 additions as the kernels
    fx = torch.floor(torch.nan_to_num(means[..., 0], nan=0.0)).clamp(-2**31, 2**31 - 1).long() - 4
    fy = torch.floor(torch.nan_to_num(means[..., 1], nan=0.0)).clamp(-2**31, 2**31 - 1).long() - 4
    wy, wx = torch.meshgrid(torch.arange(9, device=dev), torch.arange(9, device=dev), indexing="ij")
    X = fx[..., None, None] + wx; Y = fy[..., None, None] + wy    # [E,H,W,9,9]
    ok = (X >= 0) & (X < W) & (Y >= 0) & (Y < H)
    flat = merged.reshape(E, H, W, H * W)
    idx = (Y.clamp(0, H - 1) * W + X.clamp(0, W - 1)).reshape(E, H, W, 81)
    ref = torch.where(ok.reshape(E, H, W, 81), flat.gather(3, idx), torch.zeros((), device=dev))
    assert torch.equal(got[6], ref)                              # (also for out-of-box taps: re-read from the finished slices)
    a = ops.build_backward_gauss(means, covs, den, pyr[0], list(gl), 4)
    b = ops.build_backward_gauss(means, covs, den, pyr[0], None, 4, window=got[6])
    for k, (u, v) in enumerate(zip(a, b)):
        assert torch.equal(torch.nan_to_num(u), torch.nan_to_num(v)), f"gauss output {k}"
    # ... and folded into the launch itself (lgu_corr_lookup_fused_backward_gauss)
    fused = ops.corr_lookup_fused_backward(pyr, coords, off0, off1, mask, g_corr, cum_mask=cum, gauss_head=(means, covs, den))
    assert len(fused) == 9
    for k in (4, 5):
        assert torch.equal(fused[k], want[k]), f"output {k}"
    ref_g = ops.build_backward_gauss(means, covs, den, pyr[0], list(fused[:4]), 4)   # from the fused call's OWN level gradients
    for k in range(4):
        if big:
            assert (fused[k] - want[k]).abs().max().item() <= 1e-5 * max(1.0, want[k].abs().max().item())
        else:
            assert torch.equal(fused[k], want[k]), f"output {k}"
    for k, (u, v) in enumerate(zip(ref_g, fused[6:])):
        assert torch.equal(torch.nan_to_num(u), torch.nan_to_num(v)), f"fused gauss output {k}"


@pytest.mark.parametrize("keep_corr,half", [(True, False), (False, False), (False, True)])
def test_fused_lookup_with_corr_encoder_epilogue(ops, keep_corr, half):
    """SURVEY 8f-4: UpdateModule.corr_encoder[0:2] (Conv2d(196,128,1) + ReLU, droid_net.py:74-76,115) folded into the
    lookup kernel.  corr (when kept) is bit-identical to the plain fused lookup; enc agrees with F.conv2d + relu evaluated
    in fp32 (TF32 off) on that corr within 1e-5 * max(1, max|enc|); the fp16 output is that value rounded to nearest
    (compared at 1 fp16 ulp)."""
    dev = "cuda"
    E = 3
    g = inputs.gen(101)
    pyr = [torch.randn(E, 48, 64, 48 >> l, 64 >> l, generator=g).to(dev) for l in range(4)]
    c = _case(E, 102)
    coords, off0, off1 = c["coords"].to(dev), c["offsets"][0].to(dev), c["offsets"][1].to(dev)
    torch.manual_seed(5)
    conv = torch.nn.Conv2d(196, 128, 1).to(dev)
    with torch.no_grad():
        conv.weight.mul_(3.0)                                    # O(1) outputs, live low-order bits
    cum_a, cum_b = torch.ones(E, 48, 64, device=dev), torch.ones(E, 48, 64, device=dev)
    want_corr = ops.corr_lookup_fused(pyr, coords, off0, off1, 3, cum_mask=cum_a)
    frag = ops.pack_conv1x1(conv.weight)
    corr, enc = ops.corr_lookup_fused_enc(pyr, coords, off0, off1, cum_b, frag, conv.bias.detach().contiguous(), relu=True,
                                          keep_corr=keep_corr, enc_half=half)
    assert torch.equal(cum_a, cum_b)
    if keep_corr:
        assert torch.equal(corr, want_corr)
    else:
        assert corr is None
    prev = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            want = torch.relu(torch.nn.functional.conv2d(want_corr.double(), conv.weight.double(), conv.bias.double()))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    assert enc.shape == (E, 128, 48, 64) and enc.dtype == (torch.float16 if half else torch.float32)
    scale = max(1.0, want.abs().max().item())
    err = (enc.double() - want).abs().max().item()
    if half:
        assert err <= 2.0 ** -10 * scale, f"fp16 enc: {err} (scale {scale})"
    else:
        assert err <= 1e-5 * scale, f"enc: {err} (scale {scale})"


def test_backward_entry_points_refuse_mismatched_shapes_before_any_launch(ops):
    """The kernels size their reads and writes from pyramid[0]'s [E,H,W] and from f1: corr_lookup_fused_backward must
    refuse a pyramid level that is not [E,H,W,H>>l,W>>l] and build_backward_fmaps an f2 that is not f1's shape, with
    nothing launched.  The tensors are oversized, so a launch that went ahead would stay inside them."""
    import lgu_slam_b200
    E, H, W, dev = 1, 16, 32, "cuda"
    pyr = [torch.zeros(E, H, W, H >> l, W >> l, device=dev) for l in range(4)]
    coords = torch.zeros(E, H, W, 2, device=dev)
    off0, off1 = torch.zeros(E, H, W, 98, device=dev), torch.zeros(E, H, W, 98, device=dev)
    mask, g_corr = torch.ones(E, H, W, device=dev), torch.zeros(E, 196, H, W, device=dev)
    f1 = torch.zeros(E, 128, H, W, device=dev)
    launches = lgu_slam_b200._lib.LAUNCHES
    for l, shape in ((1, (E, H, W, H // 2 + 1, W // 2)), (0, (E, H, W, H + 1, W))):
        bad = list(pyr)
        bad[l] = torch.zeros(shape, device=dev)
        with pytest.raises(RuntimeError, match=rf"pyramid\[{l}\]"):
            ops.corr_lookup_fused_backward(bad, coords, off0, off1, mask, g_corr)
    with pytest.raises(RuntimeError, match="f2"):
        ops.build_backward_fmaps([torch.zeros_like(p) for p in pyr], f1, torch.zeros(E, 128, H + 2, W, device=dev))
    assert lgu_slam_b200._lib.LAUNCHES == launches

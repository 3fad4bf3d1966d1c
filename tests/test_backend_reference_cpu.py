"""tests/backend_ref.py (the float64 statement of AltCorrBlock.corr_fn that the materialised backend lookup is judged by)
against the CPU oracle's operators, composed the way corr_fn composes them (corr.py:186-215): altcorr_forward r = 1 on
level 1 -> sigmoid(var) -> offset[1] * mask -> lowMem_defSample on each of the four levels.  Small grids, no GPU."""
import pytest
import torch
import torch.nn.functional as F

import inputs
from backend_ref import backend_reference, own_masks


def _case(seed, T, N, H, W, probes):
    g = inputs.gen(seed)
    fmaps = torch.randn(T, 128, H, W, generator=g).half().float()          # fp16-valued, like the backend's buffer
    cur = fmaps / 4.0
    pyramid = []
    for l in range(4):
        if l:
            cur = F.avg_pool2d(cur, 2, stride=2)
        pyramid.append(cur.permute(0, 2, 3, 1).contiguous())             # [T,h,w,C]
    ii, jj = inputs.edge_list(T, N, g)
    coords = inputs.make_coords(N, H, W, H, W, g, probes=probes).permute(0, 2, 3, 1).contiguous()
    off0 = (4 * torch.tanh(torch.randn(N, H, W, 98, generator=g))).contiguous()
    off1 = ((4 * torch.tanh(torch.randn(N, H, W, 98, generator=g)) + off0) / 2).contiguous()
    return pyramid, ii.long(), jj.long(), coords, off0, off1


def _oracle_corr_fn(oracle, pyramid, ii, jj, coords, off0, off1, strict_ref):
    """AltCorrBlock.corr_fn's non-materialised path (corr.py:186-215) on the oracle's operators: [N,196,H,W] and the
    masked offset[1] (before the sampler zeroes its centre taps in place, quirk Q5)."""
    N, H, W, _ = coords.shape
    f1 = pyramid[0][ii].contiguous()
    offset = [off0.clone(), off1.clone(), torch.zeros_like(off0), torch.zeros_like(off0)]
    out, masked = [], None
    for i in range(4):
        f2 = pyramid[i][jj].contiguous()
        ci = (coords / 2 ** i).view(N, 1, H, W, 2).contiguous()
        if i == 1:
            m, = oracle.altcorr_forward(f1, f2, ci, 1)
            m = m.permute(0, 1, 3, 4, 2).contiguous().view(N, H, W, 3, 3)
            offset[1] = offset[1] * torch.sigmoid(torch.var(m, dim=[3, 4])).view(N, H, W, 1)
            masked = offset[1].clone()
        corr, = oracle.lowMem_defSample(f1, f2, ci, offset[i].contiguous().view(N, H, W, 7, 7, 2), 3,
                                        strict_ref=strict_ref)
        out.append(corr.view(N, 49, H, W))
    return torch.cat(out, 1), masked


def _agree(got, want, scale, slack, bar):
    gn, wn = torch.isnan(got), torch.isnan(want)
    assert torch.equal(gn, wn), f"NaN patterns differ at {int((gn != wn).sum())} values"
    ok = ~wn
    err = ((got[ok].double() - want[ok]).abs() - slack[ok]).clamp(min=0.0)
    s = scale[ok]
    bad = err > bar * s
    assert not bad.any(), f"{int(bad.sum())} values beyond {bar} S (max err/S {float((err / s.clamp(min=1e-300)).max()):.3g})"


@pytest.mark.parametrize("probes", [False, True])
@pytest.mark.parametrize("strict_ref", [True, False])
@pytest.mark.parametrize("grid", [(8, 16), (16, 8), (8, 24)])
def test_reference_matches_oracle_composition(oracle, grid, strict_ref, probes):
    H, W = grid
    T, N = 5, 4
    pyramid, ii, jj, coords, off0, off1 = _case(7 + H + W, T, N, H, W, probes)
    want, want_off1 = _oracle_corr_fn(oracle, pyramid, ii, jj, coords, off0, off1, strict_ref)
    ref, scale, slack, ref_off1 = backend_reference(pyramid, ii, jj, coords, off0, off1, strict_ref)
    P = H * W
    got = want.view(N, 196, P).permute(0, 2, 1).reshape(N * P, 196)
    if probes:
        assert torch.isnan(got).any(), "the probes should produce NaN values"
    _agree(got, ref, scale, slack, 1e-5)
    assert (scale[~torch.isnan(ref)] > 0).any()
    # the masked level-1 offsets: the slab's (edge 0's) under strict_ref, each edge's own otherwise
    mine = own_masks(pyramid, ii, jj, coords, torch.arange(N).repeat_interleave(P), torch.arange(P).repeat(N))
    left = (off1.double().view(N * P, 98) * mine.view(-1, 1)).float().view(N, P, 98)
    slab = ref_off1.view(N, P, 98)
    if strict_ref:
        assert torch.equal(slab.view(torch.int32), slab[:1].expand_as(slab).view(torch.int32))
    want_slab = left[:1].expand_as(slab) if strict_ref else left
    assert torch.allclose(slab, want_slab, rtol=1e-7, atol=0, equal_nan=True)
    # ... and the oracle's fp32 mask chain leaves fp32(offset[1] * mask) to within 1e-6 relative
    lo = want_off1.view(N, P, 98)
    assert torch.equal(torch.isnan(lo), torch.isnan(left))
    d = torch.nan_to_num((lo - left).abs() / left.abs().clamp(min=1.0), nan=0.0)
    assert d.max().item() <= 1e-6


def test_reference_sample_subsets_equal_the_full_evaluation(oracle):
    """Evaluating at chosen (edge, pixel) samples gives the same bits as the full evaluation at those samples."""
    H, W, T, N = 8, 16, 5, 3
    pyramid, ii, jj, coords, off0, off1 = _case(3, T, N, H, W, True)
    full, fs, fl, _ = backend_reference(pyramid, ii, jj, coords, off0, off1, True)
    g = inputs.gen(4)
    e = torch.randint(0, N, (40,), generator=g)
    p = torch.randint(0, H * W, (40,), generator=g)
    part, ps, pl, _ = backend_reference(pyramid, ii, jj, coords, off0, off1, True, e=e, p=p, chunk=7)
    k = e * H * W + p
    assert torch.equal(torch.nan_to_num(part, nan=7.0), torch.nan_to_num(full[k], nan=7.0))
    assert torch.equal(ps.nan_to_num(nan=7.0), fs[k].nan_to_num(nan=7.0))
    assert torch.equal(pl, fl[k])


def test_reference_helpers_follow_the_samplers_integer_semantics():
    from backend_ref import f2i, wrap
    v = torch.tensor([float("nan"), float("inf"), -float("inf"), 2147483648.0, -2147483904.0, 1e10, -3.0, 5.0])
    assert f2i(torch.floor(v)).tolist() == [0, 2 ** 31 - 1, -2 ** 31, 2 ** 31 - 1, -2 ** 31, 2 ** 31 - 1, -3, 5]
    assert wrap(torch.tensor([2 ** 31 - 1 + 1, -2 ** 31 - 1, 5])).tolist() == [-2 ** 31, 2 ** 31 - 1, 5]

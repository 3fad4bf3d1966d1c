"""AltCorrBlock.lookup_encoded: the backend lookup with update_op's corr_encoder[0:2] = relu(Conv2d(196, 128, 1)) folded
into the kernel, evaluated as the consumer evaluates it under fp16 autocast (factor_graph.py:281-286): corr, W and b
rounded to fp16, products exact, fp32 accumulation, one rounding of the output, relu keeping NaN."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import inputs

pytestmark = pytest.mark.gpu

H, W, T, E = 48, 64, 6, 5


def _setup(seed=0, probes=False):
    from importlib import import_module
    import lgu_slam_b200  # noqa: F401  (loads the library)
    corr = import_module("lgu-slam_b200.corr")
    dev = "cuda"
    torch.manual_seed(seed)
    ofsMap = nn.Conv2d(256, 98, 3, padding=1).to(dev)
    ofs_residual = nn.Conv2d(256, 98, 3, padding=1).to(dev)
    GA = corr.GaussianMask(H, W).to(dev)
    enc_net = nn.Sequential(nn.Conv2d(196, 128, 1), nn.ReLU(inplace=True), nn.Conv2d(128, 128, 3, padding=1),
                            nn.ReLU(inplace=True)).to(dev)
    with torch.no_grad():
        enc_net[0].bias.normal_(0, 0.5)              # a bias that actually moves values across zero
    g = inputs.gen(100 + seed)
    fmaps = torch.randn(1, T, 128, H, W, generator=g).half().to(dev)      # the backend's fp16 buffer (depth_video.py:36)
    ii = torch.tensor([0, 1, 2, 3, 4], device=dev)
    jj = torch.tensor([1, 2, 3, 4, 5], device=dev)
    coords = inputs.make_coords(E, H, W, H, W, g, probes=probes).permute(0, 2, 3, 1).contiguous().view(1, E, H, W, 2)
    return corr, ofsMap, ofs_residual, GA, enc_net, fmaps, ii, jj, coords.to(dev)


def _block(corr, ofsMap, ofs_residual, GA, fmaps, strict_ref=True, mode="boxes"):
    kw = dict(strict_ref=strict_ref, materialize=True)
    if mode == "cache":
        kw.update(cache=True, volume_cache_gb=1.0)
    else:
        kw.update(compact_boxes=(mode == "boxes"))
    return corr.AltCorrBlock(ofsMap, ofs_residual, GA, fmaps, **kw)


def _ordered(h):
    """fp16 -> integers ordered like the values (+0 and -0 both 0), so that a difference of 1 is one ulp."""
    b = h.contiguous().view(torch.int16).to(torch.int32)
    return torch.where(b < 0, -(b & 0x7FFF), b)


def _ulp16(v):
    """One fp16 ulp at magnitude v (fp64 tensor)."""
    e = torch.floor(torch.log2(v.clamp(min=2.0 ** -14)))
    return torch.exp2(e - 10)


def _within_one_ulp(got, want, scale, rounded=None):
    """got, want fp16.  Identical NaN patterns; elsewhere at most 1 fp16 ulp apart, or closer than the fp32 accumulation
    error at the scale of the summed terms (`scale` = sum |w16 x16| + |b16| per value; 2^-18 of it is below one fp16 ulp
    except where the terms cancel to a result near zero, and no fp32 accumulation order can do better there).
    rounded: magnitudes that `want` additionally rounded to fp16 on its way (one more ulp of those is allowed)."""
    gn, wn = torch.isnan(got), torch.isnan(want)
    assert torch.equal(gn, wn), f"NaN patterns differ at {int((gn != wn).sum())} values"
    ok = ~wn
    ulps = (_ordered(got[ok]) - _ordered(want[ok])).abs()
    tol = scale[ok] * 2.0 ** -18
    if rounded is not None:
        tol = tol + _ulp16(rounded[ok])
    slack = (got[ok].double() - want[ok].double()).abs() <= tol
    bad = (ulps > 1) & ~slack
    assert not bad.any(), f"{int(bad.sum())} values beyond 1 ulp (max {int(ulps.max())} ulp)"


def _fp64_reference(corr196, conv):
    """relu(W16 . fp16(corr) + b16) in fp64; the per-value scale sum |W16 x16| + |b16|; |W16 . fp16(corr)|."""
    x = corr196.half().double()                                    # [E,196,H,W]
    w = conv.weight.detach().half().double().view(128, 196)
    b = conv.bias.detach().half().double()
    wx = torch.einsum("ok,ekhw->eohw", w, x)
    scale = torch.einsum("ok,ekhw->eohw", w.abs(), x.abs()) + b.abs().view(1, 128, 1, 1)
    return (torch.relu(wx + b.view(1, 128, 1, 1)).half(), torch.nan_to_num(scale, nan=0.0),
            torch.nan_to_num(wx.abs(), nan=0.0))


@pytest.mark.parametrize("probes", [False, True])
@pytest.mark.parametrize("mode", ["boxes", "dense", "cache"])
@pytest.mark.parametrize("strict_ref", [True, False])
def test_lookup_encoded_matches_autocast_semantics(strict_ref, mode, probes):
    corr, ofsMap, ofs_residual, GA, enc_net, fmaps, ii, jj, coords = _setup(1, probes)
    with torch.no_grad():
        blk = _block(corr, ofsMap, ofs_residual, GA, fmaps, strict_ref, mode)
        c196 = blk(coords, ii, jj)[0]                                      # [E,196,H,W] fp32
        got = blk.lookup_encoded(coords, ii, jj, enc_net)
        assert got.shape == (1, E, 128, H, W) and got.dtype == torch.float16
        got = got[0]
        if probes:
            assert torch.isnan(c196).any(), "the probe coordinates should produce NaN rows"
        want, scale, wx = _fp64_reference(c196, enc_net[0])
        _within_one_ulp(got, want, scale)
        # torch's autocast conv: the same bar, plus one fp16 rounding of W.x (its fp16 conv need not add the bias before
        # rounding, and near a zero result that second rounding is worth up to an ulp of |W.x|)
        with torch.autocast("cuda", torch.float16):
            ac = torch.relu(F.conv2d(c196, enc_net[0].weight, enc_net[0].bias))
        assert ac.dtype == torch.float16
        _within_one_ulp(got, ac, scale, rounded=wx)
        # the first conv alone is accepted too, and gives the same bits
        assert torch.equal(blk.lookup_encoded(coords, ii, jj, enc_net[0])[0].view(torch.int16), got.view(torch.int16))


@pytest.mark.parametrize("mode", ["boxes", "dense"])
def test_lookup_encoded_writes_rows_at_out_index(mode):
    corr, ofsMap, ofs_residual, GA, enc_net, fmaps, ii, jj, coords = _setup(2)
    rows = torch.tensor([7, 0, 3, 8, 2], dtype=torch.int32, device="cuda")
    untouched = [r for r in range(9) if r not in rows.tolist()]
    with torch.no_grad():
        blk = _block(corr, ofsMap, ofs_residual, GA, fmaps, strict_ref=False, mode=mode)
        want = blk.lookup_encoded(coords, ii, jj, enc_net)[0]
        b16 = torch.full((9, 128, H, W), -7.0, dtype=torch.float16, device="cuda")
        b32 = torch.full((9, 128, H, W), -7.0, dtype=torch.float32, device="cuda")
        assert blk.lookup_encoded(coords, ii, jj, enc_net, out=b16, out_index=rows) is b16
        assert blk.lookup_encoded(coords, ii, jj, enc_net, out=b32, out_index=rows, pass_edges=2) is b32
    assert torch.equal(b16[rows.long()].view(torch.int16), want.view(torch.int16))
    assert torch.equal(b32[rows.long()].half().view(torch.int16), want.view(torch.int16))   # fp32 rows, rounded once
    assert (b16[untouched] == -7.0).all() and (b32[untouched] == -7.0).all()


@pytest.mark.parametrize("mode", ["boxes", "cache"])
@pytest.mark.parametrize("strict_ref", [True, False])
def test_lookup_encoded_leaves_the_offsets_call_leaves(strict_ref, mode):
    corr, ofsMap, ofs_residual, GA, enc_net, fmaps, ii, jj, coords = _setup(3, probes=True)
    with torch.no_grad():
        blk = _block(corr, ofsMap, ofs_residual, GA, fmaps, strict_ref, mode)
        blk(coords, ii, jj)
        want = [o.clone() for o in blk.offset]
        first = blk.lookup_encoded(coords, ii, jj, enc_net)
        got = [o.clone() for o in blk.offset]
        again = blk.lookup_encoded(coords, ii, jj, enc_net)
    assert len(got) == len(want)
    for a, b in zip(got, want):
        assert a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))
    if mode == "cache":
        assert torch.equal(again.view(torch.int16), first.view(torch.int16))


def test_lookup_encoded_rejects_what_it_does_not_implement():
    from lgu_slam_b200 import ops
    corr, ofsMap, ofs_residual, GA, enc_net, fmaps, ii, jj, coords = _setup(4)
    with torch.no_grad():
        blk = _block(corr, ofsMap, ofs_residual, GA, fmaps, strict_ref=False, mode="dense")
        with pytest.raises(RuntimeError):
            blk.lookup_encoded(coords, ii, jj, nn.Conv2d(196, 128, 3, padding=1).cuda())
        with pytest.raises(RuntimeError):
            blk.lookup_encoded(coords, ii, jj, nn.Conv2d(196, 64, 1).cuda())
        plain = corr.AltCorrBlock(ofsMap, ofs_residual, GA, fmaps, materialize=False)
        with pytest.raises(RuntimeError):
            plain.lookup_encoded(coords, ii, jj, enc_net)
        n = E * 128 * H * W
        for dtype in (torch.float16, torch.float32):
            odd = torch.empty(n + 1, dtype=dtype, device="cuda")[1:].view(E, 128, H, W)     # 2 / 4 bytes off alignment
            with pytest.raises(RuntimeError):
                blk.lookup_encoded(coords, ii, jj, enc_net, out=odd)
        with pytest.raises(RuntimeError):                                      # 196-channel rows are not encoder rows
            blk.lookup_encoded(coords, ii, jj, enc_net, out=torch.empty(E, 196, H, W, dtype=torch.float16, device="cuda"))
        # the operator: misaligned packed operands
        packed = ops.pack_conv1x1_f16(enc_net[0].weight.float(), enc_net[0].bias.float())
        odd = torch.empty(packed.numel() + 8, dtype=torch.uint8, device="cuda")[8:]
        odd.copy_(packed)
        c = coords.view(E, H, W, 2).contiguous()
        o = torch.zeros(E, H, W, 98, device="cuda")
        vols = [torch.zeros(E, H, W, H >> l, W >> l, device="cuda") for l in range(4)]
        with pytest.raises(RuntimeError):
            ops.altcorr_lookup_encoded(vols, c, o, o.clone(), 3, packed=odd)
        with pytest.raises(RuntimeError):
            ops.pack_conv1x1_f16(torch.zeros(64, 196, device="cuda"))

"""The materialised backend lookup (AltCorrBlock(materialize=True): build_boxes / build_volume / altcorr_lookup_fused /
altcorr_lookup_encoded) at N = 300 edges, against the float64 statement of corr_fn in tests/backend_ref.py.

300 edges are two passes (256 + 44) and several waves of the persistent lookup grid.  With dense level-0 volumes (the
per-chunk cache, or sparse rows for an fp32 buffer) edge e of a pass starts at e * 9.4e6 elements: edges >= 114 lie past
2^32 bytes and edges >= 228 past 2^31 elements, so every offset computation of those kernels is exercised past 32 bits.
Peak memory stays below ~18 GB (the dense cached case holds ~15 GB of volumes)."""
import time

import pytest
import torch
import torch.nn as nn

import inputs
from backend_ref import backend_reference, own_masks

pytestmark = pytest.mark.gpu

H, W, T, N = 48, 64, 24, 300
P = H * W
FULL_EDGES = (0, 1, 113, 114, 227, 228, 255, 256, 257, 299)   # pass and 2^32-byte / 2^31-element boundaries
PROBE_EDGES = (0, 228)
BAR = 2.0 ** -16
CACHE_GB = 15.0               # holds both passes' volumes (300 x 50.1 MB = 14.0 GiB)


@pytest.fixture(scope="module", autouse=True)
def _exact_torch():
    """fp32 convolutions and matmuls without TF32, and deterministic cuDNN algorithms: the offset heads then give the
    same bits for the same batch, so the reference can be fed the block's own pre-mask offsets."""
    saved = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic,
             torch.backends.cudnn.benchmark)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.benchmark = False
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    torch.cuda.synchronize()
    print(f"\n[backend scale] module time {time.perf_counter() - t0:.1f} s, peak allocated "
          f"{torch.cuda.max_memory_allocated() / 2**30:.2f} GiB")
    (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic,
     torch.backends.cudnn.benchmark) = saved


def _backend_edges(n, g):
    """Proximity-style edges like the benchmark's backend workload: every edge links a frame to one within +-8."""
    ii = torch.randint(0, T, (n,), generator=g)
    jj = (ii + torch.randint(-8, 9, (n,), generator=g)).clamp(0, T - 1)
    jj = torch.where(jj == ii, (ii + 1).clamp(max=T - 1), jj)
    jj = torch.where(jj == ii, ii - 1, jj)
    return ii, jj


def _probe(c, e, first):
    """NaN / inf / 2^31 / border probes in pixels first .. first + 15 of edge e (c [N,H,W,2])."""
    vals = [float("nan"), float("inf"), -float("inf"), 1e10, -1e10, 2147483648.0, -2147483904.0, -0.0, 0.0, -1e-30,
            float(W), float(W) - 1e-4, -1.0, -0.5]
    flat = c[e].view(-1, 2)
    for k, v in enumerate(vals):
        flat[first + k, k % 2] = v
    flat[first + len(vals)] = float("nan")


@pytest.fixture(scope="module")
def setup():
    import lgu_slam_b200  # noqa: F401  (loads the library)
    from importlib import import_module
    corr = import_module("lgu-slam_b200.corr")
    dev = "cuda"
    torch.manual_seed(20)
    ofsMap = nn.Conv2d(256, 98, 3, padding=1).to(dev)
    ofs_residual = nn.Conv2d(256, 98, 3, padding=1).to(dev)
    GA = corr.GaussianMask(H, W).to(dev)
    enc = nn.Conv2d(196, 128, 1).to(dev)
    with torch.no_grad():
        enc.bias.normal_(0, 0.5)                    # a bias that moves values across zero
    g = inputs.gen(300)
    fmaps32 = torch.randn(1, T, 128, H, W, generator=g)
    ii, jj = _backend_edges(N, g)
    c = inputs.make_coords(N, H, W, H, W, g).permute(0, 2, 3, 1).contiguous()
    _probe(c, PROBE_EDGES[0], 0)
    _probe(c, PROBE_EDGES[1], P - 15)               # the last row, in the edge past 2^31 elements of its pass
    # the samples compared with the reference: every pixel of FULL_EDGES, 64 pixels of every other edge
    corners = [0, W - 1, P - W, P - 1]
    borders = [x for k in (5, 17, 40) for x in (k, P - W + k, k * W, k * W + W - 1) if x < P]
    es, ps = [], []
    for e in range(N):
        if e in FULL_EDGES:
            px = torch.arange(P)
        else:
            px = torch.cat([torch.tensor(corners + borders), torch.randperm(P, generator=g)[:64 - 4 - len(borders)]])
        es.append(torch.full_like(px, e))
        ps.append(px)
    return dict(corr=corr, ofsMap=ofsMap, ofs_residual=ofs_residual, GA=GA, enc=enc,
                fmaps16=fmaps32.half().to(dev), fmaps32=fmaps32.to(dev), ii=ii.to(dev), jj=jj.to(dev),
                coords=c.view(1, N, H, W, 2).to(dev), e=torch.cat(es).to(dev), p=torch.cat(ps).to(dev))


def _block(s, strict_ref, mode):
    """boxes: fp16 buffer, level 0 as compact per-pixel boxes (the default); rows: fp32 buffer (hi/lo planes), level 0 as
    sparse volume rows; cache: fp16 buffer, dense volumes of both passes kept by the per-chunk cache."""
    kw = dict(strict_ref=strict_ref, materialize=True)
    if mode == "cache":
        kw.update(cache=True, volume_cache_gb=CACHE_GB)
    fm = s["fmaps32"] if mode == "rows" else s["fmaps16"]
    blk = s["corr"].AltCorrBlock(s["ofsMap"], s["ofs_residual"], s["GA"], fm, **kw)
    assert blk.materialize
    return blk


def _release():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _bits(t):
    return t.contiguous().view(torch.int16 if t.dtype == torch.float16 else torch.int32)


def _worst(got, ref, scale, slack):
    """Identical NaN patterns required; returns max over the other values of (|got - ref| - slack)+ / S."""
    gn, rn = torch.isnan(got), torch.isnan(ref)
    assert torch.equal(gn, rn), f"NaN patterns differ at {int((gn != rn).sum())} values"
    ok = ~rn
    excess = ((got[ok].double() - ref[ok]).abs() - slack[ok]).clamp(min=0.0)
    s = scale[ok]
    ratio = torch.where(excess == 0, torch.zeros_like(excess), excess / s)    # S = 0 leaves no room at all
    return float(ratio.max()) if ratio.numel() else 0.0


def _sampled(out, s):
    """[1,N,C,H,W] -> [M,C] at the samples."""
    x = out[0].reshape(N, out.shape[2], P)
    return x[s["e"], :, s["p"]]


# ------------------------------------------------------------------------------------------------
# against float64
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["boxes", "rows", "cache"])
@pytest.mark.parametrize("strict_ref", [True, False])
def test_backend_lookup_matches_fp64_at_300_edges(setup, strict_ref, mode):
    s = setup
    ii, jj, coords = s["ii"], s["jj"], s["coords"]
    with torch.no_grad():
        blk = _block(s, strict_ref, mode)
        got = blk(coords, ii, jj)
        assert got.shape == (1, N, 196, H, W)
        got = _sampled(got, s)
        # the pre-mask offsets the block sampled with: its own offset heads on the same edge batch
        n_off = blk.offset[0].shape[0]
        assert n_off == (1 if (mode == "cache" and strict_ref) else N)
        offs = blk._gen_offsets(ii[:n_off], jj[:n_off])
        assert torch.equal(_bits(offs[0].float()), _bits(blk.offset[0].float()))
        left = blk.offset[1].reshape(n_off, P, 98)
        ref, scale, slack, off1m = backend_reference(blk.pyramid, ii, jj, coords[0], offs[0].float(), offs[1].float(),
                                                     strict_ref, s["e"], s["p"], chunk=2048)
    assert torch.isnan(got).any() and (got != 0).any()
    worst = _worst(got, ref, scale, slack)
    raw = torch.nan_to_num((got.double() - ref).abs() / scale, nan=0.0)
    print(f"\n[backend scale] strict_ref={strict_ref} {mode}: max err/S {worst:.3g} (bar {BAR:.3g}); "
          f"levels 0, 2, 3 without slack {float(torch.cat((raw[:, :49], raw[:, 98:]), 1).max()):.3g}; "
          f"{int((raw > BAR).sum())} of {raw.numel()} values need the level-1 position slack")
    assert worst <= BAR
    # the offset[1] the block leaves behind: fp32(offset[1] * mask) with each edge's own mask, or the shared slab
    if n_off == 1:
        sel = s["e"] == 0
        want, have = off1m[sel], left[0, s["p"][sel]]
    else:
        m = own_masks(blk.pyramid, ii, jj, coords[0], s["e"], s["p"])
        want = (offs[1].float().reshape(n_off, P, 98)[s["e"], s["p"]].double() * m.view(-1, 1)).float()
        have = left[s["e"], s["p"]]
    assert torch.equal(torch.isnan(have), torch.isnan(want))
    d = torch.nan_to_num((have - want).abs() / want.abs().clamp(min=1.0), nan=0.0)
    assert d.max().item() <= 1e-6
    del blk, got, ref, scale, slack
    _release()


def test_the_bar_rejects_near_misses(setup):
    """The bar is tight enough to see a reference evaluated with hi-only fp16 planes of an fp32 buffer, and one with dx
    and 1 - dx swapped on one level (torch only)."""
    s = setup
    ii, jj, coords = s["ii"], s["jj"], s["coords"]
    sel = (s["e"] == 1) | (s["e"] == 2)
    e, p = s["e"][sel], s["p"][sel]
    with torch.no_grad():
        blk = _block(s, False, "rows")
        offs = [o.float() for o in blk._gen_offsets(ii, jj)]
        ref, scale, slack, _ = backend_reference(blk.pyramid, ii, jj, coords[0], offs[0], offs[1], False, e, p)
        hi = [t.half().float() for t in blk.pyramid]
        near, _, _, _ = backend_reference(hi, ii, jj, coords[0], offs[0], offs[1], False, e, p)
        w_hi = _worst(near, ref, scale, slack)
        for lvl in (0, 1, 2):
            sw, _, _, _ = backend_reference(blk.pyramid, ii, jj, coords[0], offs[0], offs[1], False, e, p, swap_dx_level=lvl)
            w_sw = _worst(sw, ref, scale, slack)
            print(f"\n[backend scale] dx swapped on level {lvl}: max err/S {w_sw:.3g}")
            assert w_sw > 16 * BAR
    print(f"\n[backend scale] hi-only planes: max err/S {w_hi:.3g}")
    assert w_hi > BAR
    del blk
    _release()


# ------------------------------------------------------------------------------------------------
# plumbing: pass schedules and destinations give the same bits
# ------------------------------------------------------------------------------------------------
def _ship_schedule():
    from importlib import import_module
    sh = import_module("lgu-slam_b200.sharded")
    sched = sh.ShardedBackendCorr._ship_schedule(N, last=True)
    assert sum(sched) == N and len(sched) > 2
    return sched


def _expected_passes(sched):
    if sched is None:
        return [(0, 256), (256, N)]
    sizes = [sched] * (-(-N // sched)) if isinstance(sched, int) else list(sched)
    bounds, a = [], 0
    for n in sizes:
        bounds.append((a, min(N, a + n)))
        a += n
    return bounds


def _plumbing(call, base, C):
    """call(**kw) -> [1,N,C,H,W] or the out buffer; base: the plain call's result."""
    for sched in (None, 37, _ship_schedule()):
        passes = []
        r = call(pass_edges=sched, pass_hook=lambda a, b: passes.append((a, b)))
        assert passes == _expected_passes(sched), (sched, passes)
        assert torch.equal(_bits(r), _bits(base)), f"pass schedule {sched} changed the result"
        del r
    g = inputs.gen(5)
    rows = torch.randperm(N + 5, generator=g)[:N].to(torch.int32).cuda()
    untouched = sorted(set(range(N + 5)) - set(rows.tolist()))
    b32 = torch.full((N + 5, C, H, W), -7.0, dtype=torch.float32, device="cuda")
    assert call(out=b32, out_index=rows) is b32
    b16 = torch.full((N + 5, C, H, W), -7.0, dtype=torch.float16, device="cuda")
    assert call(out=b16, out_index=rows, pass_edges=_ship_schedule()) is b16
    return b32, b16, rows, untouched


@pytest.mark.parametrize("strict_ref", [True, False])
def test_backend_plumbing_is_bit_identical_at_300_edges(setup, strict_ref):
    s = setup
    ii, jj, coords = s["ii"], s["jj"], s["coords"]
    with torch.no_grad():
        blk = _block(s, strict_ref, "boxes")
        base = blk(coords, ii, jj)
        b32, b16, rows, untouched = _plumbing(lambda **kw: blk(coords, ii, jj, **kw), base, 196)
    base = base[0]
    assert torch.equal(_bits(b32[rows.long()]), _bits(base))
    assert torch.equal(_bits(b16[rows.long()]), _bits(base.half()))
    assert (b32[untouched] == -7.0).all() and (b16[untouched] == -7.0).all()
    del blk, base, b32, b16
    _release()


# ------------------------------------------------------------------------------------------------
# lookup_encoded at the same N (the bar of test_backend_encoder_gpu.py, restated)
# ------------------------------------------------------------------------------------------------
def _ordered(h):
    """fp16 -> integers ordered like the values (+0 and -0 both 0), so that a difference of 1 is one ulp."""
    b = h.contiguous().view(torch.int16).to(torch.int32)
    return torch.where(b < 0, -(b & 0x7FFF), b)


def _within_one_ulp(got, want, scale):
    """got, want fp16: identical NaN patterns; elsewhere at most 1 fp16 ulp apart, or closer than the fp32 accumulation
    error at the scale of the summed terms (scale = sum |w16 x16| + |b16| per value)."""
    gn, wn = torch.isnan(got), torch.isnan(want)
    assert torch.equal(gn, wn), f"NaN patterns differ at {int((gn != wn).sum())} values"
    ok = ~wn
    ulps = (_ordered(got[ok]) - _ordered(want[ok])).abs()
    slack = (got[ok].double() - want[ok].double()).abs() <= scale[ok] * 2.0 ** -18
    bad = (ulps > 1) & ~slack
    assert not bad.any(), f"{int(bad.sum())} values beyond 1 ulp (max {int(ulps.max())} ulp)"


def _fp64_encoded(corr196, conv):
    """relu(W16 . fp16(corr) + b16) in fp64, rounded to fp16, and the per-value scale sum |W16 x16| + |b16|."""
    x = corr196.half().double()
    w = conv.weight.detach().half().double().view(128, 196)
    b = conv.bias.detach().half().double()
    wx = torch.einsum("ok,ekhw->eohw", w, x)
    scale = torch.einsum("ok,ekhw->eohw", w.abs(), x.abs()) + b.abs().view(1, 128, 1, 1)
    return torch.relu(wx + b.view(1, 128, 1, 1)).half(), torch.nan_to_num(scale, nan=0.0)


@pytest.mark.parametrize("strict_ref", [True, False])
def test_backend_lookup_encoded_at_300_edges(setup, strict_ref):
    s = setup
    ii, jj, coords, enc = s["ii"], s["jj"], s["coords"], s["enc"]
    full = torch.tensor(FULL_EDGES, device="cuda")
    with torch.no_grad():
        blk = _block(s, strict_ref, "boxes")
        c196 = blk(coords, ii, jj)[0][full]
        base = blk.lookup_encoded(coords, ii, jj, enc)
        assert base.shape == (1, N, 128, H, W) and base.dtype == torch.float16
        want, scale = _fp64_encoded(c196, enc)
        assert torch.isnan(want).any()
        _within_one_ulp(base[0][full], want, scale)
        del c196, want, scale
        b32, b16, rows, untouched = _plumbing(lambda **kw: blk.lookup_encoded(coords, ii, jj, enc, **kw), base, 128)
    base = base[0]
    assert torch.equal(_bits(b16[rows.long()]), _bits(base))
    assert torch.equal(_bits(b32[rows.long()].half()), _bits(base))       # fp32 rows, rounded once
    assert (b32[untouched] == -7.0).all() and (b16[untouched] == -7.0).all()
    del blk, base, b32, b16
    _release()


# ------------------------------------------------------------------------------------------------
# the per-chunk volume cache across pass schedules; coords that do not match the volumes
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("strict_ref", [True, False])
def test_cached_volumes_follow_the_pass_schedule(setup, strict_ref):
    """A cached block called for the same chunk (same key) with different pass schedules reuses only volumes built for
    the same edge range.  Compared with the block's first call: under strict_ref a cached block runs its offset heads
    on a batch of 1 edge, so its cuDNN rounding may differ from an uncached block's."""
    s = setup
    ii, jj, coords = s["ii"], s["jj"], s["coords"]
    budget = int(CACHE_GB * 2**30)
    with torch.no_grad():
        blk = _block(s, strict_ref, "cache")
        first = blk(coords, ii, jj, key=("chunk", 0))
        assert 0 < blk._vol_bytes <= budget
        for sched in ([37] * 8 + [4], None, _ship_schedule(), None):
            again = blk(coords, ii, jj, key=("chunk", 0), pass_edges=sched)
            assert blk._vol_bytes <= budget
            assert torch.equal(_bits(again), _bits(first)), f"pass schedule {sched} after caching changed the result"
            del again
    del blk, first
    _release()


@pytest.mark.parametrize("encoded", [False, True])
def test_backend_lookups_refuse_coords_that_do_not_match_the_volumes(setup, encoded):
    import lgu_slam_b200
    ops = lgu_slam_b200.ops
    E = 3
    vols = [torch.zeros(E, H, W, H >> l, W >> l, device="cuda") for l in range(4)]
    off = torch.zeros(E, H, W, 98, device="cuda")
    kw = {}
    if encoded:
        kw["packed"] = ops.pack_conv1x1_f16(setup["enc"].weight.detach().float(), setup["enc"].bias.detach().float())
    fn = ops.altcorr_lookup_encoded if encoded else ops.altcorr_lookup_fused
    fn(vols, torch.zeros(E, H, W, 2, device="cuda"), off, off.clone(), 3, **kw)           # the right shape runs
    torch.cuda.synchronize()
    # only oversized wrong shapes: a kernel that ignored the check would still stay inside the tensor
    for shape in ((E + 1, H, W, 2), (E, H, W + 32, 2)):
        launches = lgu_slam_b200._lib.LAUNCHES
        with pytest.raises(RuntimeError):
            fn(vols, torch.zeros(shape, device="cuda"), off, off.clone(), 3, **kw)
        assert lgu_slam_b200._lib.LAUNCHES == launches

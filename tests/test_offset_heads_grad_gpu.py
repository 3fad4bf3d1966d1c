"""GPU tests of the offset heads' backward (lgu_offset_heads_backward, corr.OffsetHeads) and of the CorrBlock paths that
use it: gradients against torch autograd of the reference chain (corr.py:117-135, per_Corr_Normalization :44-51)
evaluated in float64, one-sided and hard inputs, per-edge NaN isolation, determinism, full coverage of the outputs, and
which offset path a CorrBlock takes."""
from importlib import import_module

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import inputs

pytestmark = pytest.mark.gpu

SHAPES = [(3, 98, 48, 64), (3, 16, 24, 32)]


@pytest.fixture(scope="module")
def corr():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import lgu_slam_b200  # noqa: F401  (registers the package under its importable name)
    return import_module("lgu-slam_b200.corr")


def _chain(c0, c1):
    """The reference chain in the inputs' dtype -> (off0, off1) as [E,H,W,CH] views."""
    H, W = c0.shape[2:]

    def norm(x):
        mean = x.mean(dim=[1, 2, 3], keepdim=True)
        std = torch.sqrt(x.var(dim=[1, 2, 3], unbiased=False, keepdim=True) + 1e-5)
        return (x - mean) / std
    o0 = torch.tanh(norm(c0)) * 4
    o1 = (torch.tanh(norm(F.interpolate(c1, (H, W)))) * 4 + o0) / 2
    return o0.permute(0, 2, 3, 1), o1.permute(0, 2, 3, 1)


def _grads(fn, c0, c1, g0, g1):
    """(g_c0, g_c1) of fn(c0, c1) -> (off0, off1) for upstream gradients g0, g1 (None: that output is not used)."""
    a, b = c0.detach().clone().requires_grad_(), c1.detach().clone().requires_grad_()
    outs = fn(a, b)
    used = [(o, g) for o, g in zip(outs, (g0, g1)) if g is not None]
    ga, gb = torch.autograd.grad([o for o, _ in used], [a, b], [g.to(o.dtype) for o, g in used], allow_unused=True)
    return tuple(torch.zeros_like(x) if gx is None else gx for x, gx in zip((a, b), (ga, gb)))


def _ref(c0, c1, g0, g1):
    return _grads(_chain, c0.double(), c1.double(), g0, g1)


def _fused(corr, c0, c1, g0, g1):
    return _grads(corr.OffsetHeads.apply, c0, c1, g0, g1)


def _inputs(E, CH, H, W, seed):
    g = inputs.gen(seed)
    c0 = torch.randn(E, CH, H, W, generator=g) * 1.7 + 0.3
    c1 = torch.randn(E, CH, H // 2, W // 2, generator=g) * 0.6 - 0.2
    g0 = torch.randn(E, H, W, CH, generator=g)
    g1 = torch.randn(E, H, W, CH, generator=g)
    return [t.cuda() for t in (c0, c1, g0, g1)]


def _assert_close(got, ref, what):
    scale = max(1.0, ref.abs().max().item())
    err = (got.double() - ref).abs().max().item()
    assert err <= 1e-5 * scale, f"{what}: max err {err:.3e}, max |ref| {scale:.3e}"


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_gradients_match_the_fp64_reference_chain(corr, shape):
    c0, c1, g0, g1 = _inputs(*shape, seed=51)
    off0, off1 = corr.OffsetHeads.apply(c0, c1)
    want0, want1 = corr.ops.offset_heads(c0, c1)
    assert off0.is_contiguous() and off1.is_contiguous()
    assert torch.equal(off0, want0) and torch.equal(off1, want1), "forward must equal the inference operator bit for bit"
    got = _fused(corr, c0, c1, g0, g1)
    ref = _ref(c0, c1, g0, g1)
    assert got[0].shape == c0.shape and got[1].shape == c1.shape
    _assert_close(got[0], ref[0], "g_c0")
    _assert_close(got[1], ref[1], "g_c1")


@pytest.mark.parametrize("used", ["off0", "off1"])
def test_one_sided_gradients_match_the_reference_with_the_other_set_to_zero(corr, used):
    c0, c1, g0, g1 = _inputs(3, 98, 48, 64, seed=52)
    up = (g0, None) if used == "off0" else (None, g1)
    zero = (g0, torch.zeros_like(g1)) if used == "off0" else (torch.zeros_like(g0), g1)
    got = _fused(corr, c0, c1, *up)
    ref = _ref(c0, c1, *zero)
    _assert_close(got[0], ref[0], f"g_c0 ({used} only)")
    _assert_close(got[1], ref[1], f"g_c1 ({used} only)")
    if used == "off0":
        assert not got[1].any(), "off1 unused: c1 gets a zero gradient"


def test_constant_and_saturated_edges(corr):
    c0, c1, g0, g1 = _inputs(3, 98, 48, 64, seed=53)
    gen = inputs.gen(54)
    c0[0] = 0.75                                              # zero variance: sigma = sqrt(eps), z = 0
    c0[1] = (torch.randn(c0[1].shape, generator=gen) ** 5 * 1e3).cuda()     # heavy tails: |z| far beyond tanh's range
    c1[1] = (torch.randn(c1[1].shape, generator=gen) ** 5 * 1e3).cuda()
    x = c0[1].double()
    assert ((x - x.mean()) / x.std(unbiased=False)).abs().max() > 20
    got = _fused(corr, c0, c1, g0, g1)
    ref = _ref(c0, c1, g0, g1)
    for e in range(3):
        _assert_close(got[0][e], ref[0][e], f"g_c0 edge {e}")
        _assert_close(got[1][e], ref[1][e], f"g_c1 edge {e}")


def test_a_nan_stays_in_its_edge(corr):
    c0, c1, g0, g1 = _inputs(3, 98, 48, 64, seed=55)
    clean = _fused(corr, c0, c1, g0, g1)
    c0[1, 5, 10, 20] = float("nan")
    got = _fused(corr, c0, c1, g0, g1)
    ref = _ref(c0, c1, g0, g1)
    for k in range(2):
        assert torch.equal(torch.isnan(got[k][1]), torch.isnan(ref[k][1])), f"NaN pattern of output {k}, edge 1"
    assert torch.isfinite(got[1][1]).all(), "G1 reaches c1 through t1 only"
    for e in (0, 2):
        assert torch.equal(got[0][e], clean[0][e]) and torch.equal(got[1][e], clean[1][e]), f"edge {e} changed"


def test_backward_is_bit_identical_from_run_to_run(corr):
    c0, c1, g0, g1 = _inputs(8, 98, 48, 64, seed=56)
    _, _, stats = corr.ops.offset_heads(c0, c1, return_stats=True)
    a = corr.ops.offset_heads_backward(c0, c1, stats, g0, g1)
    b = corr.ops.offset_heads_backward(c0, c1, stats, g0, g1)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_backward_writes_every_output_element_and_nothing_past_them(corr):
    """Canary test: the outputs start as NaN with a NaN tail behind them; finite inputs leave no NaN inside and the tail
    untouched."""
    import lgu_slam_b200
    E, CH, H, W = 3, 98, 48, 64
    c0, c1, g0, g1 = _inputs(E, CH, H, W, seed=57)
    _, _, stats = corr.ops.offset_heads(c0, c1, return_stats=True)
    n0, n1, tail = c0.numel(), c1.numel(), 4096
    buf0 = torch.full((n0 + tail,), float("nan"), device="cuda")
    buf1 = torch.full((n1 + tail,), float("nan"), device="cuda")
    scratch = torch.empty(E * (H // 2) * (W // 32) * 4, dtype=torch.float64, device="cuda")
    lgu_slam_b200._lib.call_ext("lgu_offset_heads_backward", c0, c1, stats, g0, g1, buf0, buf1, scratch, E, CH, H, W,
                                torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert torch.isfinite(buf0[:n0]).all() and torch.isfinite(buf1[:n1]).all()
    assert torch.isnan(buf0[n0:]).all() and torch.isnan(buf1[n1:]).all()
    want = corr.ops.offset_heads_backward(c0, c1, stats, g0, g1)
    assert torch.equal(buf0[:n0].view_as(c0), want[0]) and torch.equal(buf1[:n1].view_as(c1), want[1])


def _block(corr, h, w, grad, **kw):
    torch.manual_seed(3)
    ofsMap = nn.Conv2d(256, 98, 3, padding=1).cuda()
    ofs_residual = nn.Conv2d(256, 98, 3, padding=1).cuda()
    GA = corr.GaussianMask(h, w).cuda()
    g = inputs.gen(58)
    f1 = torch.randn(1, 2, 128, h, w, generator=g).cuda()
    f2 = torch.randn(1, 2, 128, h, w, generator=g).cuda()
    with torch.set_grad_enabled(grad):
        blk = corr.CorrBlock(ofsMap, ofs_residual, GA, f1, f2, **kw)
    t = torch.cat((f1.reshape(2, 128, h, w), f2.reshape(2, 128, h, w)), dim=1)
    return blk, ofsMap, ofs_residual, t


def _raw(blk, k):
    return list.__getitem__(blk.offset, k)


def test_training_corrblock_with_fused_lookups_uses_the_differentiable_heads(corr):
    blk, ofsMap, ofs_residual, t = _block(corr, 48, 64, True)
    for k in (0, 1):
        o = _raw(blk, k)
        assert "OffsetHeads" in type(o.grad_fn).__name__ and o.is_contiguous() and o.shape == (2, 48, 64, 98)
    with torch.no_grad():
        want = corr.ops.offset_heads(ofsMap(t), ofs_residual(F.avg_pool2d(t, 2, 2)))
    assert torch.equal(_raw(blk, 0), want[0]) and torch.equal(_raw(blk, 1), want[1])


@pytest.mark.parametrize("case", ["per_op_lookups", "grid_30x40"])
def test_other_training_paths_keep_the_torch_chain_views(corr, case):
    if case == "per_op_lookups":
        blk, *_ = _block(corr, 48, 64, True, fused_lookup=False)
    else:
        blk, *_ = _block(corr, 30, 40, True)
    for k in (0, 1):
        o = _raw(blk, k)
        assert "Permute" in type(o.grad_fn).__name__ and not o.is_contiguous()


def test_inference_offsets_are_unchanged(corr):
    blk, ofsMap, ofs_residual, t = _block(corr, 48, 64, False)
    with torch.no_grad():
        want = corr.ops.offset_heads(ofsMap(t), ofs_residual(F.avg_pool2d(t, 2, 2)))
    for k in (0, 1):
        assert _raw(blk, k).grad_fn is None and torch.equal(_raw(blk, k), want[k])

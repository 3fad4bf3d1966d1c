"""GPU tests of the offset heads' 3x3 convolutions on the library's kernels (ops.conv3x3 / conv3x3_backward, the
lgu_conv3x3_* entry points, corr.OffsetConv): forward, input, weight and bias gradients against F.conv2d and autograd in
float64, exact power-of-two scaling, zero padding at the corners, non-finite inputs, determinism, full coverage of the
outputs, the module's fall-back to nn.Conv2d, and CorrBlock training with OffsetConv heads."""
import copy
import math
from importlib import import_module

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import inputs

pytestmark = pytest.mark.gpu

GRIDS = [(48, 64), (24, 32)]


@pytest.fixture(scope="module")
def corr():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import lgu_slam_b200  # noqa: F401  (registers the package under its importable name)
    return import_module("lgu-slam_b200.corr")


def _case(E, H, W, seed, C_in=256, C_out=98):
    """x, weight, bias (nn.Conv2d's default init range), g_y on the GPU."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    bound = 1.0 / math.sqrt(C_in * 9)
    x = torch.randn(E, C_in, H, W, generator=g, device="cuda")
    w = (torch.rand(C_out, C_in, 3, 3, generator=g, device="cuda") * 2 - 1) * bound
    b = (torch.rand(C_out, generator=g, device="cuda") * 2 - 1) * bound
    gy = torch.randn(E, C_out, H, W, generator=g, device="cuda")
    return x, w, b, gy


def _ref(x, w, b, gy):
    """F.conv2d and its autograd in float64 -> (y, g_x, g_w, g_b)."""
    xd, wd, bd = (t.double().requires_grad_() for t in (x, w, b))
    y = F.conv2d(xd, wd, bd, padding=1)
    gx, gw, gb = torch.autograd.grad(y, (xd, wd, bd), gy.double())
    return y.detach(), gx, gw, gb


def _err(got, want):
    return (got.double() - want).abs().max().item()


def _bar(want):                                    # DESIGN (c): activations and their gradients
    return 1e-5 * max(1.0, want.abs().max().item())


def _param_bar(want, N):                           # DESIGN (c): gradients of learned parameters, N positions
    return max(1e-5, 8 * 2.0 ** -24 * math.sqrt(N)) * want.abs().max().item()


def _check_all(corr, E, H, W, seed):
    x, w, b, gy = _case(E, H, W, seed)
    y = corr.ops.conv3x3(x, w, b)
    gx, gw, gb = corr.ops.conv3x3_backward(x, w, gy)
    ry, rgx, rgw, rgb = _ref(x, w, b, gy)
    assert _err(y, ry) <= _bar(ry), ("forward", _err(y, ry))
    assert _err(gx, rgx) <= _bar(rgx), ("input gradient", _err(gx, rgx))
    N = E * H * W
    assert _err(gw, rgw) <= _param_bar(rgw, N), ("weight gradient", _err(gw, rgw))
    assert _err(gb, rgb) <= _param_bar(rgb, N), ("bias gradient", _err(gb, rgb))


@pytest.mark.parametrize("E", [1, 3])
@pytest.mark.parametrize("grid", GRIDS)
def test_forward_and_gradients_match_float64(corr, E, grid):
    _check_all(corr, E, *grid, seed=11 + E)


def test_forward_and_gradients_match_float64_at_96_edges(corr):
    _check_all(corr, 96, 48, 64, seed=5)


def test_only_the_requested_gradients_are_computed(corr):
    x, w, b, gy = _case(2, 24, 32, 21)
    full = corr.ops.conv3x3_backward(x, w, gy)
    for need in ((True, False, False), (False, True, False), (False, False, True), (False, True, True)):
        got = corr.ops.conv3x3_backward(x, w, gy, *need)
        for g, want, n in zip(got, full, need):
            assert (g is None) != n and (g is None or torch.equal(g, want))


@pytest.mark.parametrize("grid", GRIDS)
def test_power_of_two_scaling_is_exact(corr, grid):
    x, w, b, gy = _case(2, *grid, 23)
    zero = torch.zeros_like(b)
    sx, sg = 2.0 ** -20, 2.0 ** -40
    y = corr.ops.conv3x3(x, w, zero)
    gx, gw, gb = corr.ops.conv3x3_backward(x, w, gy)
    assert torch.equal(corr.ops.conv3x3(x * sx, w, zero), y * sx)
    gx2, gw2, gb2 = corr.ops.conv3x3_backward(x * sx, w, gy * sg)
    assert torch.equal(gx2, gx * sg)
    assert torch.equal(gw2, gw * (sx * sg))
    assert torch.equal(gb2, gb * sg)


@pytest.mark.parametrize("grid", GRIDS)
def test_corner_impulses_reach_only_their_neighbourhood(corr, grid):
    H, W = grid
    _, w, _, _ = _case(1, H, W, 29)
    zero = torch.zeros(w.shape[0], device="cuda")
    for y0, x0 in ((0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1)):
        x = torch.zeros(1, 256, H, W, device="cuda")
        x[0, 17, y0, x0] = 1.5
        x[0, 200, y0, x0] = -0.75
        y = corr.ops.conv3x3(x, w, zero)
        ref = F.conv2d(x.double(), w.double(), padding=1)
        hood = torch.zeros(H, W, dtype=torch.bool, device="cuda")
        hood[max(0, y0 - 1):y0 + 2, max(0, x0 - 1):x0 + 2] = True
        assert (y[0][:, ~hood] == 0).all(), (y0, x0)
        assert (y[0][:, hood] != 0).all(), (y0, x0)
        assert _err(y, ref) <= _bar(ref), (y0, x0)


@pytest.mark.parametrize("grid", GRIDS)
def test_a_nan_reaches_exactly_its_neighbourhood_in_its_edge(corr, grid):
    H, W = grid
    x, w, b, _ = _case(3, H, W, 31)
    for y0, x0 in ((5, 7), (0, W - 1)):
        xn = x.clone()
        xn[0, 40, y0, x0] = float("nan")
        y = corr.ops.conv3x3(xn, w, b)
        want = torch.zeros_like(y, dtype=torch.bool)
        want[0, :, max(0, y0 - 1):y0 + 2, max(0, x0 - 1):x0 + 2] = True
        assert torch.equal(torch.isnan(y), want), (y0, x0)


def test_an_inf_gives_inf_or_nan_exactly_where_float64_does(corr):
    H, W = 48, 64
    x, w, b, _ = _case(2, H, W, 37)
    w = w.clone()
    w[3, 9, 1, 1] = 0.0          # inf * 0: NaN at the centre tap of channel 3
    w[4, 9, 0, 0] = 0.5          # exact in tf32 (its lo part is 0): still +-inf
    w[5, 9, 2, 1] = -0.25
    for y0, x0 in ((20, 30), (0, 0), (H - 1, W - 1)):
        xi = x.clone()
        xi[0, 9, y0, x0] = float("inf")
        y = corr.ops.conv3x3(xi, w, b)
        ref = F.conv2d(xi.double(), w.double(), b.double(), padding=1)
        assert torch.equal(torch.isnan(y), torch.isnan(ref)), (y0, x0)
        assert torch.equal(torch.isinf(y), torch.isinf(ref)), (y0, x0)
        inf = torch.isinf(ref)
        assert inf.any() and torch.equal(y[inf].double(), ref[inf])
        fin = torch.isfinite(ref)
        assert (y[fin].double() - ref[fin]).abs().max().item() <= _bar(ref[fin])


def test_results_are_bit_identical_from_run_to_run(corr):
    x, w, b, gy = _case(3, 48, 64, 41)
    a = (corr.ops.conv3x3(x, w, b),) + corr.ops.conv3x3_backward(x, w, gy)
    c = (corr.ops.conv3x3(x, w, b),) + corr.ops.conv3x3_backward(x, w, gy)
    for u, v in zip(a, c):
        assert torch.equal(u, v)


@pytest.mark.parametrize("grid", GRIDS)
def test_every_output_element_is_written_and_nothing_past_them(corr, grid):
    """Canary test: outputs start as NaN with a NaN tail behind them; finite inputs leave no NaN inside and the tail
    untouched, and the values equal the operator layer's."""
    import lgu_slam_b200
    L = lgu_slam_b200._lib
    H, W = grid
    E, C_in, C_out, tail = 3, 256, 98, 4096
    x, w, b, gy = _case(E, H, W, 43)
    st = torch.cuda.current_stream().cuda_stream
    nbytes = L.call_ext("lgu_conv3x3_workspace_bytes", E, C_in, C_out, H, W)
    ws = torch.full((nbytes // 4,), float("nan"), device="cuda")

    def buf(n):
        return torch.full((n + tail,), float("nan"), device="cuda")
    y, gx, gw, gb = buf(E * C_out * H * W), buf(x.numel()), buf(w.numel()), buf(C_out)
    x_hi, x_lo = corr.ops._conv3x3_planes(x)
    gy_hi, gy_lo = corr.ops._conv3x3_planes(gy)
    L.call_ext("lgu_conv3x3_forward", x_hi, x_lo, w, b, y, ws, nbytes, E, C_in, C_out, H, W, st)
    L.call_ext("lgu_conv3x3_backward_input", gy_hi, gy_lo, w, gx, ws, nbytes, E, C_in, C_out, H, W, st)
    L.call_ext("lgu_conv3x3_backward_weight", x_hi, x_lo, gy, gw, gb, ws, nbytes, E, C_in, C_out, H, W, st)
    torch.cuda.synchronize()
    want = (corr.ops.conv3x3(x, w, b),) + corr.ops.conv3x3_backward(x, w, gy)
    for got, ref in zip((y, gx, gw, gb), want):
        n = ref.numel()
        assert torch.isfinite(got[:n]).all() and torch.isnan(got[n:]).all()
        assert torch.equal(got[:n].view_as(ref), ref)


# ---------------------------------------------------------------------------------------------------------------------
# the module
# ---------------------------------------------------------------------------------------------------------------------
def _pair(corr, seed=3):
    torch.manual_seed(seed)
    ref = nn.Conv2d(256, 98, 3, padding=1).cuda()
    mod = corr.OffsetConv(256, 98).cuda()
    mod.load_state_dict(ref.state_dict())
    return ref, mod


def test_module_loads_a_conv2d_state_dict_and_takes_the_library_path(corr):
    ref, mod = _pair(corr)
    assert set(mod.state_dict()) == {"weight", "bias"} and isinstance(mod, nn.Conv2d)
    for H, W in GRIDS:
        x = torch.randn(2, 256, H, W, device="cuda").requires_grad_()
        y = mod(x)
        assert "OffsetConvFunction" in type(y.grad_fn).__name__
        assert torch.equal(y, corr.ops.conv3x3(x.detach(), mod.weight.detach(), mod.bias.detach()))


@pytest.mark.parametrize("case", ["autocast", "fp16", "fp64", "cpu", "grid_30x40"])
def test_module_falls_back_to_conv2d_bit_for_bit(corr, case):
    ref, mod = _pair(corr)
    x = torch.randn(2, 256, 48, 64, device="cuda")
    if case == "fp16":
        ref, mod, x = ref.half(), mod.half(), x.half()
    elif case == "fp64":
        ref, mod, x = ref.double(), mod.double(), x.double()
    elif case == "cpu":
        ref, mod, x = ref.cpu(), mod.cpu(), x[:1, :, :24, :32].cpu()
    elif case == "grid_30x40":
        x = x[:, :, :30, :40].contiguous()
    if case == "autocast":
        with torch.autocast("cuda", dtype=torch.float16):
            got, want = mod(x), nn.Conv2d.forward(ref, x)
        assert got.dtype == torch.float16
    else:
        got, want = mod(x), nn.Conv2d.forward(ref, x)
    assert torch.equal(got, want)
    assert got.grad_fn is None or "OffsetConvFunction" not in type(got.grad_fn).__name__


def test_module_gradients_flow_to_its_parameters(corr):
    ref, mod = _pair(corr, 4)
    x = torch.randn(3, 256, 24, 32, device="cuda", requires_grad=True)
    gy = torch.randn(3, 98, 24, 32, device="cuda")
    mod(x).backward(gy)
    rx, rw, rb = _ref(x.detach(), ref.weight.detach(), ref.bias.detach(), gy)[1:]
    assert _err(x.grad, rx) <= _bar(rx)
    assert _err(mod.weight.grad, rw) <= _param_bar(rw, 3 * 24 * 32)
    assert _err(mod.bias.grad, rb) <= _param_bar(rb, 3 * 24 * 32)


class _Float64Conv(nn.Conv2d):
    """nn.Conv2d(256, 98, 3, padding=1) evaluated in float64 (fp32 in and out): the reference heads for the offsets.
    cuDNN's own fp32 algorithms for this shape are not accurate enough to serve as one at the offsets' bar."""

    def forward(self, x):
        return F.conv2d(x.double(), self.weight.double(), self.bias.double(), padding=1).float()


class _Float64Backward(torch.autograd.Function):
    """Forward: the library's values.  Backward: autograd of F.conv2d in float64."""

    @staticmethod
    def forward(ctx, x, w, b, ops):
        ctx.save_for_backward(x, w, b)
        return ops.conv3x3(x, w, b)

    @staticmethod
    def backward(ctx, g_y):
        x, w, b = ctx.saved_tensors
        with torch.enable_grad():
            xd, wd, bd = (t.detach().double().requires_grad_() for t in (x, w, b))
            y = F.conv2d(xd, wd, bd, padding=1)
            gx, gw, gb = torch.autograd.grad(y, (xd, wd, bd), g_y.double())
        return gx.float(), gw.float(), gb.float(), None


class _Float64BackwardConv(nn.Conv2d):
    def forward(self, x):
        from importlib import import_module
        return _Float64Backward.apply(x, self.weight, self.bias, import_module("lgu-slam_b200.ops"))


def _corrblock_runs(corr, head_types):
    """CorrBlock at 48x64 (fused build and lookups), 3 edges, 3 lookups, TF32 off, once per head type, all with the same
    parameters -> per run: offsets after construction and every gradient."""
    dev = "cuda"
    torch.manual_seed(7)
    params = [nn.Conv2d(256, 98, 3, padding=1).to(dev).state_dict() for _ in range(2)]
    GA0 = corr.GaussianMask(48, 64).to(dev)
    with torch.no_grad():
        GA0.meanMap.weight.normal_(0, 0.3)
        GA0.meanMap.bias.normal_(0, 0.3)
    g = inputs.gen(61)
    b, n = 1, 3
    f1 = torch.randn(b, n, 128, 48, 64, generator=g).to(dev)
    f2 = torch.randn(b, n, 128, 48, 64, generator=g).to(dev)
    coords = [inputs.make_coords(n, 48, 64, 48, 64, g).permute(0, 2, 3, 1).contiguous().view(b, n, 48, 64, 2).to(dev)
              for _ in range(3)]
    weights = [torch.randn(b, n, 196, 48, 64, generator=g).to(dev) for _ in range(3)]
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    runs = []
    try:
        for make in head_types:
            heads = [make(corr).to(dev) for _ in range(2)]
            for h, sd in zip(heads, params):
                h.load_state_dict(sd)
            GA = copy.deepcopy(GA0)
            a, c = f1.clone().requires_grad_(), f2.clone().requires_grad_()
            blk = corr.CorrBlock(heads[0], heads[1], GA, a, c)
            offs = [list.__getitem__(blk.offset, k).detach().clone() for k in (0, 1)]
            loss = 0
            for co, wt in zip(coords, weights):
                out, mean_n, theta = blk(co)
                loss = loss + (out * wt).sum() + mean_n.sum() + theta.sum()
            loss.backward()
            runs.append(dict(offs=offs, f1=a.grad, f2=c.grad, ga={k: p.grad for k, p in GA.named_parameters()},
                             heads=[(h.weight.grad, h.bias.grad) for h in heads]))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    return runs


def test_corrblock_offsets_with_offset_conv_heads_match_float64_conv2d_heads(corr):
    ref, new = _corrblock_runs(corr, (lambda c: _Float64Conv(256, 98, 3, padding=1), lambda c: c.OffsetConv(256, 98)))
    for k in (0, 1):
        assert _err(new["offs"][k], ref["offs"][k].double()) <= _bar(ref["offs"][k]), f"offset {k}"


def test_corrblock_training_gradients_with_offset_conv_heads_match_float64_conv2d_backward(corr):
    """The same training step with OffsetConv heads and with heads whose backward is F.conv2d's in float64.  The reference
    heads' forward returns the library's values, so both blocks sample at identical positions: a lookup's gradient with
    respect to its offsets jumps where a sample crosses a cell boundary, and any difference in the offsets, however small,
    can move a sample across one."""
    ref, new = _corrblock_runs(corr, (lambda c: _Float64BackwardConv(256, 98, 3, padding=1),
                                      lambda c: c.OffsetConv(256, 98)))
    for k in (0, 1):
        assert torch.equal(new["offs"][k], ref["offs"][k])
    for k in ("f1", "f2"):
        assert _err(new[k], ref[k].double()) <= _bar(ref[k]), k
    N = 3 * 48 * 64
    for k, r in ref["ga"].items():
        if r is not None:
            assert _err(new["ga"][k], r.double()) <= _param_bar(r, N), k
    for (nw, nb), (rw, rb), npos in zip(new["heads"], ref["heads"], (N, N // 4)):
        assert _err(nw, rw.double()) <= _param_bar(rw, npos)
        assert _err(nb, rb.double()) <= _param_bar(rb, npos)

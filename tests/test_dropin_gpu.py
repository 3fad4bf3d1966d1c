"""The drop-in claim, exercised by the REFERENCE'S OWN CALLERS (VERDICT r01 "next" #1).

`oracle/build_ref.py` stages byte-for-byte copies of /root/reference/droid_slam/modules/corr.py and
/root/reference/droid_slam/gaussianMask_cuda.py under oracle/_ref/py (git-ignored, shipped to the GPU box).  Those
unmodified modules are executed three ways in one process:

  A  reference Python on the REFERENCE extension (oracle/_ref/defCorrSample_ref*.so + altcorr_ref*.so: the
     reference's CUDA kernels recompiled unmodified for sm_100)                    -- the pin
  B  reference Python with `lgu-slam_b200/dropin/defCorrSample.py` bound to `import defCorrSample`
     (and ops.altcorr_forward as `droid_backends.altcorr_forward`)                 -- the drop-in
  C  this repo's mirror classes (lgu_slam_b200.corr.CorrBlock / AltCorrBlock / GaussianMask), per-operator and
     fused paths                                                                   -- the B200-native path

Compared: outputs over >= 3 consecutive calls (cumulative offset[1] mask, quirk Q7), the in-place offset state
(quirk Q5), and every autograd gradient (feature maps, offset heads, Gaussian head).

The whole file skips unless oracle/_ref has been built and staged.  Without it, the fused build, lookup, lookup
backward and training chain at the bench shape are judged against the float64 statement in tests/frontend_ref.py
(tests/test_frontend_scale_gpu.py), and that statement against the CPU oracle (tests/test_frontend_reference_cpu.py).

Bars (fp32): forward values of A vs B bit-exact (same torch glue, bit-exact kernels); everything else
|err| <= 1e-5 * max(1, max|reference|) -- 1e-5 abs for the O(1) quantities the contract names, the same 1e-5 relative
to the tensor's largest entry where accumulated values exceed 1 (fp32 cannot resolve 1e-5 abs beyond |v| ~ 100).
Gradients of LEARNED PARAMETERS (conv / linear weights) are cuDNN / cuBLAS reductions of those per-pixel gradients
over N = E*H*W positions; rounding-level (2^-24 relative) differences of the summands accumulate as sqrt(N), so their
bar is max(1e-5, 8 * 2^-24 * sqrt(N)) * max|reference|  (3.7e-5 at N = 6144).  Other bounds that differ (tensor-core
builds) are derived where they are used.
"""
import importlib
import os
import sys
import types

import pytest
import torch
import torch.nn as nn

import inputs

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H, W = 48, 64


# ------------------------------------------------------------------------------------------------ bindings
@pytest.fixture(scope="module")
def bind():
    from oracle import build_ref
    ref_ext = build_ref.load_ref("defCorrSample_ref")
    ref_alt = build_ref.load_ref("altcorr_ref")
    if ref_ext is None or ref_alt is None or build_ref.staged_python() is None:
        pytest.skip("oracle/_ref not built/staged (run python oracle/build_ref.py in the dev container)")
    import lgu_slam_b200
    sys.path.insert(0, os.path.join(ROOT, "lgu-slam_b200", "dropin"))
    try:
        dropin = importlib.import_module("defCorrSample")          # the module a reference user puts on sys.path
    finally:
        sys.path.pop(0)
        sys.modules.pop("defCorrSample", None)
    assert dropin.__file__.endswith(os.path.join("dropin", "defCorrSample.py"))
    backends_ours = types.SimpleNamespace(altcorr_forward=lgu_slam_b200.ops.altcorr_forward)
    A = build_ref.load_ref_python(ref_ext, ref_alt, "A")
    B = build_ref.load_ref_python(dropin, backends_ours, "B")
    C = importlib.import_module("lgu-slam_b200.corr")
    return types.SimpleNamespace(A=A, B=B, C=C, ref_ext=ref_ext, ops=lgu_slam_b200.ops)


@pytest.fixture(autouse=True)
def _exact_library_math():
    prev = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.deterministic)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.deterministic = True
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.deterministic = prev


def _heads(dev, seed):
    torch.manual_seed(seed)
    ofsMap = nn.Conv2d(256, 98, 3, padding=1).to(dev)
    ofs_residual = nn.Conv2d(256, 98, 3, padding=1).to(dev)
    return ofsMap, ofs_residual


def _ga(cls, state, dev):
    ga = cls(H, W).to(dev)
    if state is not None:
        ga.load_state_dict(state)
    return ga


def _ga_state(bind, dev, seed):
    torch.manual_seed(seed)
    ga = bind.A[1].GaussianMask(H, W).to(dev)
    with torch.no_grad():      # the reference zero-initialises meanMap; use live values so that its gradients matter
        ga.meanMap.weight.normal_(0, 0.3)
        ga.meanMap.bias.normal_(0, 0.3)
    return {k: v.clone() for k, v in ga.state_dict().items()}


def _coords(n, g, b=1):
    return inputs.make_coords(b * n, H, W, H, W, g).permute(0, 2, 3, 1).contiguous().view(b, n, H, W, 2)


def _close(got, want, what, tol=1e-5):
    want = want.float()
    scale = max(1.0, want.abs().max().item())
    err = (got.float() - want).abs().max().item()
    assert err <= tol * scale, f"{what}: max abs err {err:.3e} > {tol:g} * {scale:.3g}"
    return err / scale


def _param_tol(n_pos):
    return max(1e-5, 8 * 2.0 ** -24 * n_pos ** 0.5)


def _params(ofsMap, ofs_residual, ga):
    return [("ofsMap.weight", ofsMap.weight), ("ofsMap.bias", ofsMap.bias), ("ofs_residual.weight", ofs_residual.weight),
            ("GA.map.weight", ga.map.weight), ("GA.covMap.weight", ga.covMap.weight), ("GA.meanMap.weight", ga.meanMap.weight)]


def _run_corrblock(make_block, ga, heads, fm1, fm2, coords, wts, train):
    """One pass of the reference's usage pattern (droid_net.py:187-222): build, `len(coords)` lookups, one backward."""
    ofsMap, ofs_residual = heads
    for _, p in _params(ofsMap, ofs_residual, ga):
        p.grad = None
    f1 = fm1.clone().requires_grad_(train)
    f2 = fm2.clone().requires_grad_(train)
    with torch.set_grad_enabled(train):
        blk = make_block(ofsMap, ofs_residual, ga, f1, f2)
        outs, states, loss = [], [], 0.0
        for c, w in zip(coords, wts):
            out, mean_n, theta = blk(c)
            outs.append(out.detach().clone())
            states.append([o.detach().clone() for o in blk.offset])
            loss = loss + (out * w).sum() + (mean_n.square().sum() + theta.sum()) * 1e-2
        grads = {}
        if train:
            loss.backward()
            grads = {"fmap1": f1.grad.clone(), "fmap2": f2.grad.clone()}
            grads.update({k: p.grad.clone() for k, p in _params(ofsMap, ofs_residual, ga)})
    pyr = [t.detach() for t in blk.corr_pyramid]
    return types.SimpleNamespace(outs=outs, states=states, grads=grads, pyr=pyr, mean_n=blk.mean_n.detach(),
                                 theta=blk.theta.detach())


def _case(bind, dev, n, steps, seed, half):
    g = inputs.gen(seed)
    fm1 = torch.randn(1, n, 128, H, W, generator=g)
    fm2 = torch.randn(1, n, 128, H, W, generator=g)
    if half:
        fm1, fm2 = fm1.half().float(), fm2.half().float()
    coords = [_coords(n, g).to(dev) for _ in range(steps)]
    # upstream gradients scaled so that the accumulated feature-map gradients stay O(1)
    wts = [(torch.randn(1, n, 196, H, W, generator=g) * 0.05).to(dev) for _ in range(steps)]
    return fm1.to(dev), fm2.to(dev), coords, wts


# ------------------------------------------------------------------------------------------------ CorrBlock
@pytest.mark.parametrize("train", [False, True])
def test_reference_corrblock_runs_identically_on_the_dropin(bind, train):
    """A vs B: the reference's CorrBlock (corr.py:53-141), unmodified, on the reference extension and on the drop-in."""
    dev = "cuda"
    heads = _heads(dev, 11)
    state = _ga_state(bind, dev, 12)
    fm1, fm2, coords, wts = _case(bind, dev, n=2, steps=3, seed=13, half=not train)
    res = {}
    for tag, mods in (("A", bind.A), ("B", bind.B)):
        ga = _ga(mods[1].GaussianMask, state, dev)
        res[tag] = _run_corrblock(mods[0].CorrBlock, ga, heads, fm1, fm2, coords, wts, train)
    a, b = res["A"], res["B"]
    for l in range(4):
        assert torch.equal(a.pyr[l], b.pyr[l]), f"pyramid level {l}: gaussianMask forward must be bit-exact"
    for k in range(len(coords)):
        assert torch.equal(a.outs[k], b.outs[k]), f"lookup {k}: forward must be bit-exact"
        for l in range(4):
            assert torch.equal(a.states[k][l], b.states[k][l]), f"offset[{l}] state after call {k}"
    assert torch.equal(a.mean_n, b.mean_n) and torch.equal(a.theta, b.theta)
    if train:
        for k in a.grads:
            tol = 1e-5 if k.startswith("fmap") else _param_tol(2 * H * W)
            _close(b.grads[k], a.grads[k], f"grad {k} (drop-in vs reference extension)", tol)


@pytest.mark.parametrize("mode", ["per_op", "fused_dense", "fused_accumulate"])
def test_mirror_corrblock_training_equals_reference_graph(bind, mode):
    """C vs A: this repo's CorrBlock against the reference's CorrBlock on the reference's compiled kernels --
    outputs of every lookup and every autograd gradient.  per_op: the same op sequence on the drop-in operators;
    fused_*: FusedBuild (tcgen05, 3-term fp16 split) + FusedCorrLookup (one launch each way), level gradients returned
    densely or accumulated in persistent buffers."""
    dev = "cuda"
    heads = _heads(dev, 21)
    state = _ga_state(bind, dev, 22)
    fm1, fm2, coords, wts = _case(bind, dev, n=2, steps=3, seed=23, half=False)
    a = _run_corrblock(bind.A[0].CorrBlock, _ga(bind.A[1].GaussianMask, state, dev), heads, fm1, fm2, coords, wts, True)
    kw = dict(per_op=dict(fused=False, fused_lookup=False),
              fused_dense=dict(fused=True, fused_lookup=True, accumulate_grads=False),
              fused_accumulate=dict(fused=True, fused_lookup=True, accumulate_grads=True))[mode]
    make = lambda *args: bind.C.CorrBlock(*args, **kw)
    c = _run_corrblock(make, _ga(bind.C.GaussianMask, state, dev), heads, fm1, fm2, coords, wts, True)
    report = []
    for l in range(4):
        # fused build: fp16 hi/lo split, three MMAs -> <= 2^-21 relative per product, K = 128 terms of O(1/16): 1e-5 abs
        report.append(f"pyr{l} {_close(c.pyr[l], a.pyr[l], f'pyramid level {l}'):.2e}")
    for k in range(len(coords)):
        report.append(f"out{k} {_close(c.outs[k], a.outs[k], f'lookup {k}'):.2e}")
    _close(c.mean_n, a.mean_n, "mean_n")
    _close(c.theta, a.theta, "theta")
    for k in a.grads:
        # Feature-map gradients of the fused build: tcgen05 kind::tf32 with a 3-term hi/lo split (lo*lo dropped: 2^-22
        # relative per product) and chunked fp32 accumulation over K = 3072..4080 terms (DESIGN.md: <= 7e-6 of the result's
        # largest entry measured, 1e-5 stated) -- the same 1e-5 * max|ref| bar as every other gradient.
        tol = 1e-5 if k.startswith("fmap") else _param_tol(2 * H * W)
        report.append(f"{k} {_close(c.grads[k], a.grads[k], f'grad {k} ({mode} vs reference graph)', tol):.2e}")
    print(mode, "relative errors:", ", ".join(report))


def test_mirror_corrblock_inference_and_state_equal_reference(bind):
    """C vs A in inference (fp16-valued maps, the frontend's case): fused build + fused lookup over 3 calls; the stored
    offset[1] carries the cumulative mask like the reference's (centre tap excepted: read as 0 by both, see Q5)."""
    dev = "cuda"
    heads = _heads(dev, 31)
    state = _ga_state(bind, dev, 32)
    fm1, fm2, coords, wts = _case(bind, dev, n=3, steps=3, seed=33, half=True)
    a = _run_corrblock(bind.A[0].CorrBlock, _ga(bind.A[1].GaussianMask, state, dev), heads, fm1, fm2, coords, wts, False)
    c = _run_corrblock(bind.C.CorrBlock, _ga(bind.C.GaussianMask, state, dev), heads, fm1, fm2, coords, wts, False)
    for l in range(4):
        _close(c.pyr[l], a.pyr[l], f"pyramid level {l}")
    for k in range(len(coords)):
        _close(c.outs[k], a.outs[k], f"lookup {k}")
        d = (c.states[k][1].reshape(3, H, W, 49, 2) - a.states[k][1].reshape(3, H, W, 49, 2)).clone()
        d[..., 24, :] = 0
        assert d.abs().max().item() <= 1e-5, f"offset[1] state after call {k}"


def test_reference_cat_and_getitem_on_the_dropin(bind):
    """corr.py:111-115,137-141 make the offsets contiguous, after which the kernels' in-place centre-tap zeroing (Q5)
    reaches the block's own state -- identical on both extensions."""
    dev = "cuda"
    heads = _heads(dev, 41)
    state = _ga_state(bind, dev, 42)
    fm1, fm2, coords, _ = _case(bind, dev, n=3, steps=2, seed=43, half=True)
    res = []
    for mods in (bind.A, bind.B):
        ga = _ga(mods[1].GaussianMask, state, dev)
        with torch.no_grad():
            x = mods[0].CorrBlock(heads[0], heads[1], ga, fm1[:, :2].contiguous(), fm2[:, :2].contiguous())
            y = mods[0].CorrBlock(heads[0], heads[1], ga, fm1[:, 2:].contiguous(), fm2[:, 2:].contiguous())
            blk = x.cat(y)
            o1, _, _ = blk(coords[0])
            blk = blk[torch.tensor([True, False, True], device=dev)]
            o2, _, _ = blk(coords[1][:, [0, 2]].contiguous())
            res.append((o1, o2, [o.clone() for o in blk.offset]))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
    for l in range(4):
        assert torch.equal(res[0][2][l], res[1][2][l])
    assert res[0][2][0].view(2, H, W, 49, 2)[..., 24, :].abs().max().item() == 0      # zeroed in place after cat


# ------------------------------------------------------------------------------------------------ GaussianMask
def test_gaussianmask_module_forward_backward(bind):
    """gaussianMask_cuda.py:35-88 on both extensions and the mirror: corr1, mean, det and the MLP gradients."""
    dev = "cuda"
    state = _ga_state(bind, dev, 51)
    g = inputs.gen(52)
    E = 2
    x = torch.randn(E, H, W, 256, generator=g).to(dev)
    corr = torch.randn(E, H, W, H, W, generator=g).to(dev)
    w = (torch.randn(E, H, W, H, W, generator=g) * 0.05).to(dev)
    res = []
    for cls in (bind.A[1].GaussianMask, bind.B[1].GaussianMask, bind.C.GaussianMask):
        ga = _ga(cls, state, dev)
        xi = x.clone().requires_grad_()
        corr1, mean, det = ga(xi, corr)
        ((corr1 * w).sum() + mean.square().sum() * 1e-2 + det.sum() * 1e-2).backward()
        res.append((corr1.detach(), mean.detach(), det.detach(), xi.grad.clone(),
                    [p.grad.clone() for p in (ga.map.weight, ga.covMap.weight, ga.meanMap.weight, ga.meanMap.bias)]))
    a = res[0]
    assert torch.equal(res[1][0], a[0]) and torch.equal(res[1][1], a[1]) and torch.equal(res[1][2], a[2])
    for tag, r in (("drop-in", res[1]), ("mirror", res[2])):
        _close(r[0], a[0], f"{tag} corr1")
        _close(r[1], a[1], f"{tag} mean")
        _close(r[2], a[2], f"{tag} det")
        _close(r[3], a[3], f"{tag} grad x")
        for k, (p, q) in enumerate(zip(r[4], a[4])):
            _close(p, q, f"{tag} grad param {k}", _param_tol(E * H * W))


# ------------------------------------------------------------------------------------------------ AltCorrBlock
def _run_alt(cls, ga, heads, fmaps, chunks, coords, **kw):
    with torch.no_grad():
        blk = cls(heads[0], heads[1], ga, fmaps, **kw)
        outs, offs = [], []
        for (ii, jj), c in zip(chunks, coords):
            outs.append(blk(c, ii, jj))
            offs.append([o.clone() for o in blk.offset])
    return outs, offs


def test_reference_altcorrblock_on_the_dropin_and_the_mirror(bind):
    """corr.py:155-249 (the backend's on-the-fly path: altcorr_forward + 4 x lowMem_defSample, fp16 buffer): A vs B vs the
    mirror's two paths (drop-in operator sequence; per-level tcgen05 volumes + fused per-corner-gated lookup)."""
    dev = "cuda"
    heads = _heads(dev, 61)
    state = _ga_state(bind, dev, 62)
    g = inputs.gen(63)
    T = 6
    fmaps = torch.randn(1, T, 128, H, W, generator=g).half().to(dev)
    chunks = [(torch.tensor([0, 1, 2, 3, 4, 5, 2], device=dev), torch.tensor([1, 2, 3, 4, 5, 4, 0], device=dev)),
              (torch.tensor([5, 4, 3], device=dev), torch.tensor([0, 1, 2], device=dev))]
    coords = [_coords(ii.numel(), g).to(dev) for ii, _ in chunks]
    a_out, a_off = _run_alt(bind.A[0].AltCorrBlock, _ga(bind.A[1].GaussianMask, state, dev), heads, fmaps, chunks, coords)
    b_out, b_off = _run_alt(bind.B[0].AltCorrBlock, _ga(bind.B[1].GaussianMask, state, dev), heads, fmaps, chunks, coords)
    gaC = _ga(bind.C.GaussianMask, state, dev)
    c_out, c_off = _run_alt(bind.C.AltCorrBlock, gaC, heads, fmaps, chunks, coords, materialize=False)
    m_out, m_off = _run_alt(bind.C.AltCorrBlock, gaC, heads, fmaps, chunks, coords, materialize=True)
    for k in range(len(chunks)):
        assert a_out[k].shape == b_out[k].shape == c_out[k].shape == m_out[k].shape
        _close(b_out[k], a_out[k], f"chunk {k}: reference AltCorrBlock on the drop-in")
        _close(c_out[k], a_out[k], f"chunk {k}: mirror AltCorrBlock (operator sequence)")
        # materialised path: dot-then-interpolate on exact fp16 products vs the reference's interpolate-then-dot in fp32:
        # both sum 128 products of magnitude <= |f1||f2|/16 per tap; reassociation error <= 128 * 2^-24 * sum|terms| ~ 1e-5 * max
        _close(m_out[k], a_out[k], f"chunk {k}: mirror AltCorrBlock (tcgen05 volumes + fused lookup)", tol=2e-5)
        assert torch.equal(b_off[k][1], a_off[k][1]) or _close(b_off[k][1], a_off[k][1], "offset[1] * mask") <= 1e-5
        d = (m_off[k][1].reshape(-1, H, W, 49, 2) - a_off[k][1].reshape(-1, H, W, 49, 2)).clone()
        d[..., 24, :] = 0
        assert d.abs().max().item() <= 1e-5


# ------------------------------------------------------------------------------------------------ fused lookup backward
def _bare_block(cls, pyr, offs, n):
    """A CorrBlock around given pyramid / offset tensors (skipping __init__): what __call__ needs."""
    blk = object.__new__(cls)
    blk.num_levels, blk.radius = 4, 3
    blk.corr_pyramid = list(pyr)
    blk.offset = list(offs)
    blk.mean_n = torch.zeros(1, n, H, W, 2, device=pyr[0].device)
    blk.theta = torch.zeros(1, n, H, W, device=pyr[0].device)
    return blk


@pytest.mark.parametrize("E,steps", [(3, 3), (48, 1)])
@pytest.mark.parametrize("accumulate", [False, True])
def test_fused_lookup_backward_vs_reference_autograd(bind, E, steps, accumulate):
    """lgu_corr_lookup_fused_backward (dense) and ..._accumulate against the autograd graph of the reference's
    CorrBlock.__call__ (corr.py:88-109) on the reference's compiled kernels: gradients of the four pyramid levels and of
    both offset tensors after `steps` cumulative lookups.  E = 48 is the bench shape (frontend_w20_e48)."""
    dev = "cuda"
    g = inputs.gen(700 + E)
    pyr0 = [torch.randn(E, H, W, H >> l, W >> l, generator=g).to(dev) for l in range(4)]
    off_a = (4 * torch.tanh(torch.randn(E, 98, H, W, generator=g))).to(dev)
    off_b = ((4 * torch.tanh(torch.randn(E, 98, H, W, generator=g))).to(dev) + off_a) / 2
    coords = [_coords(E, g).to(dev) for _ in range(steps)]
    wts = [torch.randn(1, E, 196, H, W, generator=g).to(dev) for _ in range(steps)]
    res = []
    for which in ("ref", "ours"):
        pyr = [p.clone().requires_grad_() for p in pyr0]
        o0 = off_a.clone().requires_grad_()
        o1 = off_b.clone().requires_grad_()
        offs = [o0.permute(0, 2, 3, 1), o1.permute(0, 2, 3, 1)]          # permuted views, as corr.py:129-130 leaves them
        offs += [torch.zeros_like(offs[0]).detach(), torch.zeros_like(offs[0]).detach()]
        if which == "ref":
            blk = _bare_block(bind.A[0].CorrBlock, pyr, offs, E)
            use = pyr
        else:
            blk = _bare_block(bind.C.CorrBlock, pyr, offs, E)
            blk.fused_lookup, blk._gacc, blk._token = True, None, None
            use = pyr
            if accumulate:
                # the training clip's arrangement: level gradients accumulate in persistent buffers owned by the build
                acc = bind.C.LevelGradAccumulator()
                acc.levels = tuple(pyr)
                blk._gacc = acc
                blk._token = torch.zeros(1, device=dev, requires_grad=True)
        loss, outs = 0.0, []
        for c, w in zip(coords, wts):
            out, _, _ = blk(c)
            outs.append(out.detach())
            loss = loss + (out * w).sum()
        loss.backward()
        if which == "ours" and accumulate:
            gl = blk._gacc.take()
        else:
            gl = [p.grad for p in use]
        res.append((outs, [t.clone() for t in gl], o0.grad.clone(), o1.grad.clone()))
        del blk, pyr, loss
    (outs_a, gl_a, g0_a, g1_a), (outs_c, gl_c, g0_c, g1_c) = res
    for k in range(steps):
        _close(outs_c[k], outs_a[k], f"lookup {k}")
    for l in range(4):
        _close(gl_c[l], gl_a[l], f"grad pyramid level {l}")
    _close(g0_c, g0_a, "grad offset[0]")
    _close(g1_c, g1_a, "grad offset[1]")


def test_fused_lookup_forward_at_bench_shape_vs_reference_ops(bind):
    """E = 48 (frontend_w20_e48): lgu_corr_lookup_fused against the reference's five compiled operators + torch glue."""
    dev = "cuda"
    E = 48
    g = inputs.gen(801)
    pyr = [torch.randn(E, H, W, H >> l, W >> l, generator=g).to(dev) for l in range(4)]
    c = inputs.frontend_case(E=E, T=20, seed=802)
    offs = [o.to(dev) for o in c["offsets"]]
    coords = c["coords"].to(dev).view(1, E, H, W, 2)
    with torch.no_grad():
        ref_blk = _bare_block(bind.A[0].CorrBlock, pyr, [o.clone() for o in offs], E)
        want, _, _ = ref_blk(coords)
        got = bind.ops.corr_lookup_fused(pyr, coords.view(E, H, W, 2).contiguous(), offs[0].clone(), offs[1].clone(), 3)
    want = want.view(E, 196, H, W)
    for l in (0, 2, 3):
        assert torch.equal(got[:, 49 * l:49 * (l + 1)], want[:, 49 * l:49 * (l + 1)]), f"level {l} must be bit-exact"
    # level 1: its offsets carry sigmoid(var) -- a few ulp apart between torch's reduction and the kernel's -- times the
    # local slope of a white-noise pyramid (|V| up to ~5): 1e-5 relative to the largest value
    _close(got[:, 49:98], want[:, 49:98], "level 1")


@pytest.mark.parametrize("E", [4, 48])
def test_bench_step_backward_with_folded_gaussian_head_vs_reference_autograd(bind, E):
    """The backward half of bench.py's step -- lgu_corr_lookup_fused_backward_gauss: one launch that returns the level and
    offset gradients AND the Gaussian head's (means, covs, den) gradients -- against autograd through the reference's own
    Python: GaussianMaskCuda (gaussianMask_cuda.py:7-24) / den + corr (:84-86), 3 x avg_pool2d (corr.py:83-86) and
    CorrBlock.__call__ (corr.py:88-109), all on the reference's compiled kernels.  E = 48 is the bench shape."""
    dev = "cuda"
    g = inputs.gen(900 + E)
    import torch.nn.functional as F
    GaussFn = bind.A[1].GaussianMaskCuda
    raw = (torch.randn(E, H, W, H, W, generator=g) * 2).to(dev)
    ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32), indexing="ij")
    mean0 = (torch.stack([xs, ys], -1)[None] + 1.5 * torch.randn(E, H, W, 2, generator=g)).to(dev)
    mean0[0, 0, 0] = torch.tensor([-2.5, 1.25]); mean0[0, 0, 1] = torch.tensor([65.0, 49.0])     # windows over the borders
    cov0 = (torch.rand(E, H, W, 2, generator=g) * 5 + 0.05).to(dev)
    den0 = (6.28 * torch.sqrt(cov0[..., 0] * cov0[..., 1])).contiguous()
    off_a = (4 * torch.tanh(torch.randn(E, 98, H, W, generator=g))).to(dev)
    off_b = (4 * torch.tanh(torch.randn(E, 98, H, W, generator=g))).to(dev)
    coords = _coords(E, g).to(dev)
    w = (torch.randn(1, E, 196, H, W, generator=g)).to(dev)
    # ---- the reference graph
    mean, cov, den = mean0.clone().requires_grad_(), cov0.clone().requires_grad_(), den0.clone().requires_grad_()
    o0, o1 = off_a.clone().requires_grad_(), off_b.clone().requires_grad_()
    corr1 = GaussFn.apply(mean, cov, raw, 4) / den.view(E, H, W, 1, 1) + raw
    cur = corr1.reshape(E * H * W, 1, H, W)
    pyr = []
    for l in range(4):
        pyr.append(cur.view(E, H, W, H >> l, W >> l))
        cur = F.avg_pool2d(cur, 2, stride=2)
    offs = [o0.permute(0, 2, 3, 1), o1.permute(0, 2, 3, 1)]
    offs += [torch.zeros_like(offs[0]).detach(), torch.zeros_like(offs[0]).detach()]
    blk = _bare_block(bind.A[0].CorrBlock, pyr, offs, E)
    out, _, _ = blk(coords)
    (out * w).sum().backward()
    want = dict(out=out.detach(), gm=mean.grad, gc=cov.grad, gd=den.grad, g0=o0.grad, g1=o1.grad)
    # ---- ours, on the same pyramid values
    ops = bind.ops
    pyr_d = [p.detach().contiguous() for p in pyr]
    del blk, corr1, cur
    c = coords.view(E, H, W, 2).contiguous()
    a0 = off_a.permute(0, 2, 3, 1).contiguous()
    a1 = off_b.permute(0, 2, 3, 1).contiguous()
    cum = torch.ones(E, H, W, device=dev)
    corr, mask = ops.corr_lookup_fused(pyr_d, c, a0, a1, 3, return_mask=True, cum_mask=cum)
    _close(corr, want["out"].view(E, 196, H, W), "lookup")
    res = ops.corr_lookup_fused_backward(pyr_d, c, a0, a1, mask, w.view(E, 196, H, W).contiguous(), cum_mask=cum,
                                         gauss_head=(mean0.contiguous(), cov0.contiguous(), den0))
    _close(res[6], want["gm"], "grad means")
    _close(res[7], want["gc"], "grad covs")
    _close(res[8], want["gd"], "grad den")
    _close(res[4].view(E, H, W, 98).permute(0, 3, 1, 2), want["g0"], "grad offset[0]")
    _close(res[5].view(E, H, W, 98).permute(0, 3, 1, 2), want["g1"], "grad offset[1]")

"""GPU tests of the host-side mirror (lgu-slam_b200/corr.py): CorrBlock / AltCorrBlock / GaussianMask keep the
reference's interface (corr.py:53-152,155-249; gaussianMask_cuda.py:35-88) and their fused inference paths agree
with their own per-operator (autograd) paths, which in turn are the reference's op sequence on the parity-tested
operators."""
import pytest
import torch
import torch.nn as nn

import inputs

pytestmark = pytest.mark.gpu


def _modules(dev, seed=0):
    import lgu_slam_b200
    from importlib import import_module
    corr = import_module("lgu-slam_b200.corr")
    torch.manual_seed(seed)
    ofsMap = nn.Conv2d(256, 98, 3, padding=1).to(dev)
    ofs_residual = nn.Conv2d(256, 98, 3, padding=1).to(dev)
    GA = corr.GaussianMask(48, 64).to(dev)
    with torch.no_grad():      # the reference zero-initialises meanMap (droid_net.py:149-156); use live values here
        GA.meanMap.weight.normal_(0, 0.3)
        GA.meanMap.bias.normal_(0, 0.3)
    return corr, ofsMap, ofs_residual, GA


def test_corrblock_fused_inference_matches_per_op_path():
    dev = "cuda"
    corr, ofsMap, ofs_residual, GA = _modules(dev)
    g = inputs.gen(7)
    b, n = 1, 3
    fmap1 = torch.randn(b, n, 128, 48, 64, generator=g).half().float().to(dev)
    fmap2 = torch.randn(b, n, 128, 48, 64, generator=g).half().float().to(dev)
    coords = inputs.make_coords(n, 48, 64, 48, 64, g).permute(0, 2, 3, 1).contiguous().view(b, n, 48, 64, 2).to(dev)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            blk_f = corr.CorrBlock(ofsMap, ofs_residual, GA, fmap1, fmap2, fused=True)
            blk_p = corr.CorrBlock(ofsMap, ofs_residual, GA, fmap1, fmap2, fused=False)
            for l in range(4):
                assert blk_f.corr_pyramid[l].shape == (n, 48, 64, 48 >> l, 64 >> l)
                err = (blk_f.corr_pyramid[l] - blk_p.corr_pyramid[l]).abs().max().item()
                assert err <= 2e-5, f"pyramid level {l}: {err}"
            assert torch.allclose(blk_f.mean_n, blk_p.mean_n) and torch.allclose(blk_f.theta, blk_p.theta)
            # lookups: fused launch vs per-op autograd functions on the SAME pyramid
            blk_p.corr_pyramid = [t.clone() for t in blk_f.corr_pyramid]
            blk_p._can_fuse_lookup = lambda c: False
            for it in range(2):                                     # second call checks the cumulative mask (Q7)
                out_f, mean_f, theta_f = blk_f(coords)
                out_p, _, _ = blk_p(coords)
                assert out_f.shape == (b, n, 196, 48, 64)
                assert (out_f - out_p).abs().max().item() <= 1e-5, f"call {it}"
                # cumulative offset state, except the centre tap (tap 24): read as 0 by both paths, zeroed in memory
                # only by the per-op path's in-place quirk Q5
                d = (blk_f.offset[1] - blk_p.offset[1].reshape(blk_f.offset[1].shape)).view(n, 48, 64, 49, 2)
                d[..., 24, :] = 0
                assert d.abs().max().item() <= 1e-5
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def test_corrblock_on_a_grid_the_fused_kernels_do_not_cover(oracle):
    """TUM-RGBD shape (240x320 images -> 30x40 maps; odd pooled sizes 15x20 / 7x10 / 3x5): neither the tcgen05 build
    (W = 64) nor the fused lookup (W % 32 = 0) applies, so CorrBlock must run the reference's per-operator sequence on the
    drop-in kernels -- checked against the CPU oracle's composition of the reference ops on the block's own pyramid."""
    dev = "cuda"
    import lgu_slam_b200
    from importlib import import_module
    corr = import_module("lgu-slam_b200.corr")
    torch.manual_seed(3)
    ofsMap = nn.Conv2d(256, 98, 3, padding=1).to(dev)
    ofs_residual = nn.Conv2d(256, 98, 3, padding=1).to(dev)
    GA = corr.GaussianMask(30, 40).to(dev)
    g = inputs.gen(17)
    b, n, h, w = 1, 2, 30, 40
    fmap1 = torch.randn(b, n, 128, h, w, generator=g).to(dev)
    fmap2 = torch.randn(b, n, 128, h, w, generator=g).to(dev)
    coords = inputs.make_coords(n, h, w, h, w, g).permute(0, 2, 3, 1).contiguous().view(b, n, h, w, 2).to(dev)
    with torch.no_grad():
        blk = corr.CorrBlock(ofsMap, ofs_residual, GA, fmap1, fmap2)
        assert [tuple(t.shape[3:]) for t in blk.corr_pyramid] == [(30, 40), (15, 20), (7, 10), (3, 5)]
        assert not blk._can_fuse_lookup(coords)
        pyr_cpu = [t.cpu().contiguous() for t in blk.corr_pyramid]
        offs_cpu = [o.cpu().clone() for o in blk.offset]
        for it in range(2):
            out, _, _ = blk(coords)
            want = oracle.corr_block_lookup(pyr_cpu, coords.view(n, h, w, 2).cpu(), offs_cpu, 3)
            assert out.shape == (b, n, 196, h, w)
            got = out.view(n, 196, h, w).cpu()
            for l in (0, 2, 3):     # levels whose offsets do not pass through the mask: bit-exact
                assert torch.equal(got[:, 49 * l:49 * (l + 1)], want[:, 49 * l:49 * (l + 1)]), f"call {it} level {l}"
            assert (got[:, 49:98] - want[:, 49:98]).abs().max().item() <= 1e-5, f"call {it} level 1"


def test_corrblock_training_path_has_gradients():
    dev = "cuda"
    corr, ofsMap, ofs_residual, GA = _modules(dev, 1)
    g = inputs.gen(8)
    fmap1 = torch.randn(1, 2, 128, 48, 64, generator=g).to(dev).requires_grad_()
    fmap2 = torch.randn(1, 2, 128, 48, 64, generator=g).to(dev).requires_grad_()
    coords = inputs.make_coords(2, 48, 64, 48, 64, g).permute(0, 2, 3, 1).contiguous().view(1, 2, 48, 64, 2).to(dev)
    blk = corr.CorrBlock(ofsMap, ofs_residual, GA, fmap1, fmap2)
    out, mean_n, theta = blk(coords)
    assert out.shape == (1, 2, 196, 48, 64) and mean_n.shape == (1, 2, 48, 64, 2) and theta.shape == (1, 2, 48, 64)
    (out.square().mean() + mean_n.mean() + theta.mean()).backward()
    for t in (fmap1, fmap2, ofsMap.weight, ofs_residual.weight, GA.covMap.weight, GA.meanMap.weight, GA.map.weight):
        assert t.grad is not None and torch.isfinite(t.grad).all() and t.grad.abs().sum() > 0


def test_corrblock_cat_and_getitem_keep_edge_order():
    dev = "cuda"
    corr, ofsMap, ofs_residual, GA = _modules(dev, 2)
    g = inputs.gen(9)
    f1 = torch.randn(1, 3, 128, 48, 64, generator=g).half().float().to(dev)
    f2 = torch.randn(1, 3, 128, 48, 64, generator=g).half().float().to(dev)
    coords = inputs.make_coords(3, 48, 64, 48, 64, g).permute(0, 2, 3, 1).contiguous().view(1, 3, 48, 64, 2).to(dev)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False       # the offset convs: TF32 would differ between batch sizes (~1e-3)
    with torch.no_grad():
        whole = corr.CorrBlock(ofsMap, ofs_residual, GA, f1, f2)
        a = corr.CorrBlock(ofsMap, ofs_residual, GA, f1[:, :2], f2[:, :2])
        b_ = corr.CorrBlock(ofsMap, ofs_residual, GA, f1[:, 2:], f2[:, 2:])
        joined = a.cat(b_)
        o_whole, _, _ = whole(coords)
        o_join, _, _ = joined(coords)
        # per-edge normalisation of the offsets makes edges independent, so the concatenated block equals the whole
        # (up to cuDNN choosing different fp32 conv algorithms for different batch sizes)
        assert (o_whole - o_join).abs().max().item() <= 1e-3
        keep = torch.tensor([True, False, True], device=dev)
        sub = whole[keep]
        assert sub.corr_pyramid[0].shape[0] == 2 and sub.offset[1].shape[0] == 2
    torch.backends.cudnn.allow_tf32 = prev


def test_altcorrblock_interface_and_shapes(oracle):
    dev = "cuda"
    corr, ofsMap, ofs_residual, GA = _modules(dev, 3)
    g = inputs.gen(10)
    T = 5
    fmaps = torch.randn(1, T, 128, 48, 64, generator=g).half().to(dev)
    ii = torch.tensor([0, 1, 2, 3], device=dev)
    jj = torch.tensor([1, 2, 3, 4], device=dev)
    coords = inputs.make_coords(4, 48, 64, 48, 64, g).permute(0, 2, 3, 1).contiguous().view(1, 4, 48, 64, 2).to(dev)
    with torch.no_grad():
        blk = corr.AltCorrBlock(ofsMap, ofs_residual, GA, fmaps, materialize=False)
        out = blk(coords, ii, jj)
        assert out.shape == (1, 4, 196, 48, 64) and torch.isfinite(out).all()
        # zero-offset levels (2, 3) equal the oracle's lowMem sampler on the same pooled maps
        # AltCorrBlock keeps the buffer's dtype (fp16, depth_video.py:36): each pooled level is rounded to fp16
        f = fmaps.float().cpu()[0] / 4.0
        pyr = [f]
        for _ in range(3):
            pyr.append(torch.nn.functional.avg_pool2d(pyr[-1], 2, 2).half().float())
        f1 = pyr[0][ii.cpu()].permute(0, 2, 3, 1).contiguous()
        for l in (2, 3):
            f2 = pyr[l][jj.cpu()].permute(0, 2, 3, 1).contiguous()
            c = (coords.cpu()[0] / 2 ** l).view(4, 1, 48, 64, 2).contiguous()
            want, = oracle.lowMem_defSample(f1, f2, c, torch.zeros(4, 48, 64, 7, 7, 2), 3)
            got = out[0, :, 49 * l:49 * (l + 1)].cpu()
            assert (got - want.view(4, 49, 48, 64)).abs().max().item() <= 1e-4


@pytest.mark.parametrize("strict_ref", [True, False])
@pytest.mark.parametrize("half", [True, False])
def test_altcorrblock_materialized_matches_lowmem_operators(strict_ref, half):
    """The B200 backend path (per-level volumes on tcgen05 + fused per-corner-gated lookup) against the reference's
    op sequence on the drop-in operators (altcorr_forward + 4 x lowMem_defSample, themselves parity-tested against
    the oracle and the compiled reference).  Tolerance: 1e-4 abs on values of magnitude ~10 (dot-then-interpolate vs
    interpolate-then-dot in fp32; the fp16 buffer's products are exact in the tensor core)."""
    dev = "cuda"
    corr, ofsMap, ofs_residual, GA = _modules(dev, 4)
    g = inputs.gen(11)
    T, E = 6, 7
    fmaps = torch.randn(1, T, 128, 48, 64, generator=g)
    fmaps = (fmaps.half() if half else fmaps).to(dev)
    ii = torch.tensor([0, 1, 2, 3, 4, 5, 2], device=dev)
    jj = torch.tensor([1, 2, 3, 4, 5, 4, 0], device=dev)
    coords = inputs.make_coords(E, 48, 64, 48, 64, g).permute(0, 2, 3, 1).contiguous().view(1, E, 48, 64, 2).to(dev)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            a = corr.AltCorrBlock(ofsMap, ofs_residual, GA, fmaps, strict_ref=strict_ref, materialize=True)
            b = corr.AltCorrBlock(ofsMap, ofs_residual, GA, fmaps, strict_ref=strict_ref, materialize=False)
            assert a.materialize and not b.materialize
            out_a = a(coords, ii, jj)
            out_b = b(coords, ii, jj)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    assert out_a.shape == out_b.shape == (1, E, 196, 48, 64)
    assert torch.equal(out_a == 0, out_b == 0) or ((out_a == 0) ^ (out_b == 0)).float().mean().item() < 1e-4
    err = (out_a - out_b).abs().max().item()
    assert err <= 1e-4 * max(1.0, out_b.abs().max().item() / 10), f"max abs err {err} (max |v| {out_b.abs().max().item()})"
    d = (a.offset[1] - b.offset[1]).reshape(E, 48, 64, 49, 2)
    d[..., 24, :] = 0          # the centre tap: zeroed in memory only by the drop-in operator's in-place quirk (Q5)
    assert d.abs().max().item() <= 1e-5


@pytest.mark.parametrize("strict_ref", [True, False])
def test_altcorr_cache_across_ba_steps(strict_ref):
    """Global BA calls the block for the same chunk in every iteration (factor_graph.py:265-279) with new coords: the
    cached block (offset heads and volumes kept per chunk) must return what the uncached block returns, call after
    call, must be bit-reproducible, and must not let one call's mask leak into the next (the reference regenerates
    the offsets on every call, corr.py:186-189)."""
    dev = "cuda"
    corr, ofsMap, ofs_residual, GA = _modules(dev, 8)
    g = inputs.gen(21)
    T, E = 6, 7
    fmaps = torch.randn(1, T, 128, 48, 64, generator=g).half().to(dev)
    chunks = [(torch.tensor([0, 1, 2, 3, 4, 5, 2], device=dev), torch.tensor([1, 2, 3, 4, 5, 4, 0], device=dev)),
              (torch.tensor([5, 4, 3], device=dev), torch.tensor([0, 1, 2], device=dev))]
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            a = corr.AltCorrBlock(ofsMap, ofs_residual, GA, fmaps, strict_ref=strict_ref, cache=True, volume_cache_gb=1.0)
            b = corr.AltCorrBlock(ofsMap, ofs_residual, GA, fmaps, strict_ref=strict_ref, cache=False)
            assert a.materialize and b.materialize
            first = {}
            for step in range(3):
                for ci, (ii, jj) in enumerate(chunks):
                    n = ii.numel()
                    coords = inputs.make_coords(n, 48, 64, 48, 64, inputs.gen(100 + 10 * ci + (step % 2)))
                    coords = coords.permute(0, 2, 3, 1).contiguous().view(1, n, 48, 64, 2).to(dev)
                    out_a, out_b = a(coords, ii, jj), b(coords, ii, jj)
                    err = (out_a - out_b).abs().max().item()
                    assert err <= 1e-4 * max(1.0, out_b.abs().max().item() / 10), f"step {step} chunk {ci}: {err}"
                    if step == 0:
                        first[ci] = out_a.clone()
                    elif step == 2:            # same coords as step 0: two cached calls and a different one in between
                        assert torch.equal(out_a, first[ci]), "cached calls must be bit-reproducible"
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    assert len(a._cache) == 2 and a._vol_bytes == (7 + 3) * 4 * 3072 * (3072 + 768 + 192 + 48)
    a.clear_cache()
    assert not a._cache and a._vol_bytes == 0


def test_build_volume_matches_matmul(ops):
    dev = "cuda"
    g = inputs.gen(12)
    f1 = (torch.randn(3, 3072, 128, generator=g) / 4).half().to(dev)
    for Q in (3072, 768, 192, 48):
        f2 = (torch.randn(4, Q, 128, generator=g) / 4).half().to(dev)
        ii = torch.tensor([0, 2, 1, 1], dtype=torch.int32, device=dev)
        jj = torch.tensor([3, 0, 1, 2], dtype=torch.int32, device=dev)
        got = ops.build_volume(f1, None, f2, None, ii, jj)
        want = torch.matmul(f1[ii.long()].double(), f2[jj.long()].double().transpose(1, 2))
        assert got.shape == (4, 3072, Q)
        assert (got.double() - want).abs().max().item() <= 1e-5, f"Q={Q}"


def test_pooled_corrblock_matches_corrblock_through_add_and_remove():
    """Edge-slot pool (SURVEY 8f-2): build into slots, cat, drop edges, add more (reusing freed slots), look up --
    identical to the copying CorrBlock at every stage."""
    dev = "cuda"
    corr, ofsMap, ofs_residual, GA = _modules(dev, 5)
    g = inputs.gen(13)
    mk = lambda n: (torch.randn(1, n, 128, 48, 64, generator=g).half().to(dev),
                    torch.randn(1, n, 128, 48, 64, generator=g).half().to(dev))
    mc = lambda n: inputs.make_coords(n, 48, 64, 48, 64, g).permute(0, 2, 3, 1).contiguous().view(1, n, 48, 64, 2).to(dev)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            pool = corr.CorrPool(6, 48, 64, dev)
            fa, fb, fc = mk(3), mk(2), mk(2)
            ref = corr.CorrBlock(ofsMap, ofs_residual, GA, *fa)
            blk = corr.PooledCorrBlock(pool, ofsMap, ofs_residual, GA, *fa)
            ref = ref.cat(corr.CorrBlock(ofsMap, ofs_residual, GA, *fb))
            blk = blk.cat(corr.PooledCorrBlock(pool, ofsMap, ofs_residual, GA, *fb))
            assert len(blk) == 5 and len(pool.free) == 1
            c5 = mc(5)
            o_ref, _, _ = ref(c5)
            o_blk, mean_n, theta = blk(c5)
            assert torch.equal(o_ref, o_blk) and mean_n.shape == (1, 5, 48, 64, 2) and theta.shape == (1, 5, 48, 64)
            keep = torch.tensor([True, False, True, True, False], device=dev)
            ref, blk = ref[keep], blk[keep]
            assert len(blk) == 3 and len(pool.free) == 3
            ref = ref.cat(corr.CorrBlock(ofsMap, ofs_residual, GA, *fc))
            blk = blk.cat(corr.PooledCorrBlock(pool, ofsMap, ofs_residual, GA, *fc))      # reuses the freed slots
            c5b = mc(5)
            for _ in range(2):                                   # second call: cumulative offset[1] mask per slot (Q7)
                o_ref, _, _ = ref(c5b)
                o_blk, _, _ = blk(c5b)
                assert torch.equal(o_ref, o_blk)
            with pytest.raises(RuntimeError, match="slots requested"):
                corr.PooledCorrBlock(pool, ofsMap, ofs_residual, GA, *mk(2))
    finally:
        torch.backends.cudnn.allow_tf32 = prev


@pytest.mark.parametrize("accumulate", [True, False])
def test_training_clip_fused_lookup_equals_per_op_autograd(accumulate):
    """BASELINE configs[2] in miniature (train.py step shape: a clip's edges, several lookup iterations, one backward,
    droid_net.py:187-222): the same CorrBlock with the fused differentiable build + lookup (2 + 2 launches per
    iteration pair) and with the reference's per-operator autograd graph gives the same outputs and the same gradients
    on feature maps, offset heads and Gaussian head."""
    dev = "cuda"
    g = inputs.gen(14)
    b, n, steps = 2, 5, 3
    fm1 = torch.randn(b, n, 128, 48, 64, generator=g).to(dev)
    fm2 = torch.randn(b, n, 128, 48, 64, generator=g).to(dev)
    coords = [inputs.make_coords(b * n, 48, 64, 48, 64, g).permute(0, 2, 3, 1).contiguous().view(b, n, 48, 64, 2).to(dev)
              for _ in range(steps)]
    wts = [torch.randn(b, n, 196, 48, 64, generator=g).to(dev) for _ in range(steps)]
    prev = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    res = []
    try:
        for fused_lookup in (True, False):
            corr, ofsMap, ofs_residual, GA = _modules(dev, 6)
            f1, f2 = fm1.clone().requires_grad_(), fm2.clone().requires_grad_()
            # fused: differentiable tcgen05 build (FusedBuild) + differentiable fused lookup; else the reference's graph
            # accumulate: the lookups' level gradients go into persistent buffers (LevelGradAccumulator), else every
            # lookup returns dense gradients that autograd sums
            blk = corr.CorrBlock(ofsMap, ofs_residual, GA, f1, f2, fused=fused_lookup, fused_lookup=fused_lookup,
                                 accumulate_grads=accumulate)
            assert ("FusedBuild" in type(blk.corr_pyramid[0].grad_fn).__name__) == fused_lookup
            assert (blk._gacc is not None) == (fused_lookup and accumulate)
            loss = 0.0
            outs = []
            for c, w in zip(coords, wts):
                out, mean_n, theta = blk(c)
                outs.append(out.detach())
                loss = loss + (out * w * 0.05).sum() + 1e-2 * (mean_n.square().sum() + theta.sum())
            loss.backward()
            if blk._gacc is not None:
                assert blk._gacc.grads is None, "FusedBuild.backward must consume (and free) the accumulators"
            res.append((outs, [t.grad.clone() for t in (f1, f2, ofsMap.weight, ofs_residual.weight, GA.map.weight,
                                                         GA.covMap.weight, GA.meanMap.weight)]))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    (outs_a, grads_a), (outs_b, grads_b) = res
    for k, (a, bb) in enumerate(zip(outs_a, outs_b)):
        assert (a - bb).abs().max().item() <= 2e-5, f"lookup {k}"
    names = ("fmap1", "fmap2", "ofsMap.weight", "ofs_residual.weight", "GA.map.weight", "GA.covMap.weight",
             "GA.meanMap.weight")
    # the fused path -- build, lookups, their backward and the training chain's leaf gradients (maps, mean / cov / det,
    # offsets) -- is judged against an fp64 statement in tests/test_frontend_scale_gpu.py, which also checks that
    # CorrBlock(fused=True) wires its modules into those ops.  Here the two paths of this repo must agree:
    # |err| <= 1e-5 * max(1, max|per-op gradient|)
    # (learned-parameter gradients are cuDNN / cuBLAS reductions of the per-pixel gradients over N = E*H*W positions:
    # rounding-level differences of the summands accumulate as sqrt(N) -> 8 * 2^-24 * sqrt(N) relative, see test_dropin_gpu)
    n_pos = b * n * 48 * 64
    report = []
    for name, a, bb in zip(names, grads_a, grads_b):
        tol = 1e-5 if name.startswith("fmap") else max(1e-5, 8 * 2.0 ** -24 * n_pos ** 0.5)
        scale = max(1.0, bb.abs().max().item())
        err = (a - bb).abs().max().item()
        report.append(f"{name}: max err {err:.3e}, max |g| {bb.abs().max().item():.3e}")
        assert err <= tol * scale, "; ".join(report)
    print("\n".join(report))


def test_pool_build_writes_only_its_slots():
    """Canary test (compute-sanitizer is closed on this pool): the slot-indirected build writes exactly the slots it was
    given -- every other slot of the pool keeps its NaN sentinel bit pattern, and the written slots hold no sentinel."""
    dev = "cuda"
    corr, ofsMap, ofs_residual, GA = _modules(dev, 7)
    g = inputs.gen(15)
    pool = corr.CorrPool(5, 48, 64, dev)
    for t in pool.levels:
        t.fill_(float("nan"))
    pool.free = [4, 2, 0, 3, 1]                       # alloc() pops from the end: the block gets slots 1 and 3
    f1 = torch.randn(1, 2, 128, 48, 64, generator=g).half().to(dev)
    f2 = torch.randn(1, 2, 128, 48, 64, generator=g).half().to(dev)
    with torch.no_grad():
        blk = corr.PooledCorrBlock(pool, ofsMap, ofs_residual, GA, f1, f2)
    assert sorted(blk.slots) == [1, 3]
    for l, t in enumerate(pool.levels):
        assert torch.isnan(t[[0, 2, 4]]).all(), f"level {l}: a slot outside the block was written"
        assert torch.isfinite(t[[1, 3]]).all(), f"level {l}: a slot of the block was not fully written"


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_altcorrblock_writes_into_a_callers_buffer_at_given_rows(dtype):
    """The sharded backend's return path (sharded.PeerOutput): AltCorrBlock(out=, out_index=) stores edge e's rows at
    out[out_index[e]] -- fp32 bit-identical to the returned tensor, fp16 = that tensor rounded to nearest -- and leaves
    every other row of the buffer untouched."""
    dev = "cuda"
    corr, ofsMap, ofs_residual, GA = _modules(dev, 9)
    g = inputs.gen(31)
    T, E = 6, 5
    fmaps = torch.randn(1, T, 128, 48, 64, generator=g).half().to(dev)
    ii = torch.tensor([0, 1, 2, 3, 4], device=dev)
    jj = torch.tensor([1, 2, 3, 4, 5], device=dev)
    coords = inputs.make_coords(E, 48, 64, 48, 64, g).permute(0, 2, 3, 1).contiguous().view(1, E, 48, 64, 2).to(dev)
    rows = torch.tensor([7, 0, 3, 8, 2], dtype=torch.int32, device=dev)
    with torch.no_grad():
        blk = corr.AltCorrBlock(ofsMap, ofs_residual, GA, fmaps, materialize=True)
        want = blk(coords, ii, jj)[0]
        buf = torch.full((9, 196, 48, 64), -7.0, dtype=dtype, device=dev)
        ret = blk(coords, ii, jj, out=buf, out_index=rows)
    assert ret is buf
    got = buf[rows.long()]
    if dtype == torch.float32:
        assert torch.equal(got, want)
    else:
        assert torch.equal(got, want.half())
    untouched = [r for r in range(9) if r not in rows.tolist()]
    assert (buf[untouched] == -7.0).all()


def test_offset_heads_kernel_matches_the_reference_chain(ops):
    """lgu_offset_heads (2 launches) against the reference's chain (corr.py:117-135 with per_Corr_Normalization :44-51),
    evaluated by torch in fp32: offsets agree within 1e-5 (|offset| <= 4; statistics are accumulated in fp64 here and by
    Welford in torch), layout [E,H,W,98] contiguous."""
    dev = "cuda"
    g = inputs.gen(41)
    E, CH, H, W = 3, 98, 48, 64
    c0 = (torch.randn(E, CH, H, W, generator=g) * 1.7 + 0.3).to(dev)
    c1 = (torch.randn(E, CH, H // 2, W // 2, generator=g) * 0.6 - 0.2).to(dev)

    def norm(x):
        mean = x.mean(dim=[1, 2, 3], keepdim=True)
        std = torch.sqrt(x.var(dim=[1, 2, 3], unbiased=False, keepdim=True) + 1e-5)
        return (x - mean) / std
    w0 = torch.tanh(norm(c0)) * 4
    w1 = (torch.tanh(norm(torch.nn.functional.interpolate(c1, (H, W)))) * 4 + w0) / 2
    off0, off1 = ops.offset_heads(c0, c1)
    assert off0.shape == (E, H, W, CH) and off0.is_contiguous() and off1.is_contiguous()
    assert (off0 - w0.permute(0, 2, 3, 1)).abs().max().item() <= 1e-5
    assert (off1 - w1.permute(0, 2, 3, 1)).abs().max().item() <= 1e-5


def test_build_forms_the_gaussian_denominator_itself(ops):
    """den = NULL: the build kernel computes 6.28 * sqrt(cov_x * cov_y) in its prologue -- bit-identical pyramids."""
    dev = "cuda"
    c = inputs.frontend_case(E=3, T=4, seed=43)
    hi, _ = ops.pack_fmaps(c["fmaps"].half().to(dev))
    ii, jj, means, covs = c["ii"].to(dev), c["jj"].to(dev), c["means"].to(dev), c["covs"].to(dev)
    den = (6.28 * torch.sqrt(covs[..., 0] * covs[..., 1])).contiguous()
    a = ops.build_pyramid(hi, None, ii, jj, 48, 64, means=means, covs=covs, den=den, gauss_radius=4)
    b = ops.build_pyramid(hi, None, ii, jj, 48, 64, means=means, covs=covs, den=None, gauss_radius=4)
    for l in range(4):
        assert torch.equal(a[l], b[l]), f"level {l}"


def test_corrblock_lookup_encoded_matches_call_plus_corr_encoder():
    """CorrBlock.lookup_encoded (the fused lookup with UpdateModule.corr_encoder[0:2] folded in) == relu(conv1x1(__call__)),
    and both keep the block's cumulative offset state in step."""
    dev = "cuda"
    corr, ofsMap, ofs_residual, GA = _modules(dev, 10)
    g = inputs.gen(51)
    f1 = torch.randn(1, 3, 128, 48, 64, generator=g).half().to(dev)
    f2 = torch.randn(1, 3, 128, 48, 64, generator=g).half().to(dev)
    coords = [inputs.make_coords(3, 48, 64, 48, 64, g).permute(0, 2, 3, 1).contiguous().view(1, 3, 48, 64, 2).to(dev) for _ in range(2)]
    torch.manual_seed(6)
    enc_net = nn.Sequential(nn.Conv2d(196, 128, 1), nn.ReLU(inplace=True), nn.Conv2d(128, 128, 3, padding=1), nn.ReLU(inplace=True)).to(dev)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            a = corr.CorrBlock(ofsMap, ofs_residual, GA, f1, f2)
            b = corr.CorrBlock(ofsMap, ofs_residual, GA, f1, f2)
            for c in coords:
                out, _, _ = a(c)
                want = torch.relu(enc_net[0](out.view(3, 196, 48, 64)))
                kept, enc, mean_n, theta = b.lookup_encoded(c, enc_net, keep_corr=True)
                assert torch.equal(kept, out) and enc.shape == (1, 3, 128, 48, 64)
                err = (enc.view(3, 128, 48, 64) - want).abs().max().item()
                assert err <= 2e-5 * max(1.0, want.abs().max().item()), err       # both sides are fp32 evaluations here
            enc_only, _, _ = b.lookup_encoded(coords[0], enc_net[0])
            assert enc_only.shape == (1, 3, 128, 48, 64)
    finally:
        torch.backends.cudnn.allow_tf32 = prev


@pytest.mark.parametrize("probes", [False, True])
def test_sparse_volumes_are_what_the_backend_lookup_reads(probes):
    """lgu_volume_half_mask + lgu_build_volume_sparse: the halves the mask names are bit-identical to the dense build,
    and the fused backend lookup (per-corner gating, offsets bounded by 4 -- 4 * tanh, corr.py:121-128, including the
    bound itself) returns the same bits from the sparse volume although everything else in it is NaN-poisoned scratch."""
    from lgu_slam_b200 import ops
    dev, E, H, W, T = "cuda", 5, 48, 64, 4
    g = inputs.gen(77)
    fm = (torch.randn(T, 128, H, W, generator=g) / 4).half().to(dev)
    planes = []
    cur = fm.float()
    for l in range(4):
        planes.append(cur.permute(0, 2, 3, 1).reshape(T, -1, 128).half().contiguous())
        cur = torch.nn.functional.avg_pool2d(cur, 2, stride=2)
    ii = torch.tensor([0, 1, 2, 3, 1], dtype=torch.int32, device=dev)
    jj = torch.tensor([1, 2, 3, 0, 0], dtype=torch.int32, device=dev)
    coords = inputs.make_coords(E, H, W, H, W, g, probes=probes).permute(0, 2, 3, 1).contiguous().to(dev)
    off = [(4.0 * torch.tanh(3.0 * torch.randn(E, H, W, 98, generator=g))).to(dev).contiguous() for _ in range(2)]
    off[0][0, 0, :, :] = 4.0                                      # the bound itself, both signs
    off[0][0, 1, :, :] = -4.0
    off[1][1, 0, :, :] = 4.0
    dense = [ops.build_volume(planes[0], None, planes[l], None, ii, jj).view(E, H, W, H >> l, W >> l) for l in range(4)]
    hm = ops.volume_half_mask(coords, 0)
    assert hm.shape == (E * H * W // 128,)
    hm1 = ops.volume_half_mask(coords, 1)
    poison = torch.full((E, H * W, H * W), float("nan"), device=dev)
    del poison                                                    # the caching allocator hands this block to the next call
    sparse0 = ops.build_volume(planes[0], None, planes[0], None, ii, jj, half_mask=hm).view(E, H, W, H, W)
    bits = ((hm.view(E, H * W // 128, 1).long() & 0xffffffff) >> torch.arange(12, device=dev).view(1, 1, 12)) & 1   # [E,units,12]
    frac = bits.float().mean().item()
    assert 0.2 < frac < 1.0, f"mask density {frac}"
    written = bits.bool().view(E, H * W // 128, 1, 12, 1, 1).expand(E, H * W // 128, 128, 12, 4, W)
    written = written.reshape(E, H, W, H, W)
    assert torch.equal(sparse0[written], dense[0][written])
    want = ops.altcorr_lookup_fused(dense, coords, off[0], off[1].clone(), 3, shared_offsets=False, apply_mask=True)
    poison = torch.full((E, H * W, H * W // 4), float("nan"), device=dev)
    del poison
    sparse1 = ops.build_volume(planes[0], None, planes[1], None, ii, jj, half_mask=hm1).view(E, H, W, H // 2, W // 2)
    got = ops.altcorr_lookup_fused([sparse0, sparse1] + dense[2:], coords, off[0], off[1].clone(), 3, shared_offsets=False,
                                   apply_mask=True)
    assert torch.equal(torch.isnan(got), torch.isnan(want))       # (NaN only where a probe coordinate produces one)
    assert torch.equal(torch.nan_to_num(got), torch.nan_to_num(want))


@pytest.mark.parametrize("probes", [False, True])
def test_compact_level0_boxes_give_the_backend_lookup_the_same_bits(probes):
    """lgu_build_boxes + lgu_altcorr_lookup_boxes_into: level 0 kept as one 16 x 20 box per source pixel (what the fused
    backend lookup stages anyway) instead of a volume.  The boxes equal the corresponding windows of the dense volume bit
    for bit (zeros outside the grid) and the lookup returns the same bits, offsets bounded by 4 including the bound itself
    and coordinates whose sum with 4.0 rounds up to the next integer (tap on the box's last row with dy == 0)."""
    from lgu_slam_b200 import ops
    dev, E, H, W, T = "cuda", 5, 48, 64, 4
    g = inputs.gen(78)
    fm = (torch.randn(T, 128, H, W, generator=g) / 4).half().to(dev)
    planes = []
    cur = fm.float()
    for l in range(4):
        planes.append(cur.permute(0, 2, 3, 1).reshape(T, -1, 128).half().contiguous())
        cur = torch.nn.functional.avg_pool2d(cur, 2, stride=2)
    ii = torch.tensor([0, 1, 2, 3, 1], dtype=torch.int32, device=dev)
    jj = torch.tensor([1, 2, 3, 0, 0], dtype=torch.int32, device=dev)
    coords = inputs.make_coords(E, H, W, H, W, g, probes=probes).permute(0, 2, 3, 1).contiguous().to(dev)
    coords[1, 5, :, :] = torch.tensor([30.999998, 20.999998])    # + 4.0 rounds up to 35.0 / 25.0 in fp32
    coords[1, 6, :, :] = torch.tensor([10.9999995, 39.9999962])
    off = [(4.0 * torch.tanh(3.0 * torch.randn(E, H, W, 98, generator=g))).to(dev).contiguous() for _ in range(2)]
    off[0][0, 0, :, :] = 4.0
    off[0][0, 1, :, :] = -4.0
    off[0][1, 5:7, :, :] = 4.0
    off[1][1, 0, :, :] = 4.0
    dense = [ops.build_volume(planes[0], None, planes[l], None, ii, jj).view(E, H, W, H >> l, W >> l) for l in range(4)]
    poison = torch.full((E, H * W, 16, 20), float("nan"), device=dev)
    del poison
    boxes = ops.build_boxes(planes[0], planes[0], ii, jj, coords)
    assert boxes.shape == (E, H * W, 16, 20)
    # the boxes against windows of the dense volume
    c = torch.nan_to_num(coords.reshape(E, H * W, 2), nan=0.0)
    fx = torch.floor(c[..., 0]).clamp(-64, W + 64).long()
    fy = torch.floor(c[..., 1]).clamp(-64, H + 64).long()
    xb = ((fx - 7) >> 2) << 2
    yb = fy - 7
    Y = yb[..., None, None] + torch.arange(16, device=dev).view(1, 1, 16, 1)
    X = xb[..., None, None] + torch.arange(20, device=dev).view(1, 1, 1, 20)
    ok = (X >= 0) & (X < W) & (Y >= 0) & (Y < H)
    idx = (Y.clamp(0, H - 1) * W + X.clamp(0, W - 1)).reshape(E, H * W, 320)
    want_boxes = torch.where(ok.reshape(E, H * W, 320), dense[0].reshape(E, H * W, H * W).gather(2, idx),
                             torch.zeros((), device=dev)).view(E, H * W, 16, 20)
    assert torch.equal(boxes, want_boxes)
    want = ops.altcorr_lookup_fused(dense, coords, off[0], off[1].clone(), 3, shared_offsets=False, apply_mask=True)
    got = ops.altcorr_lookup_fused([None] + dense[1:], coords, off[0], off[1].clone(), 3, shared_offsets=False,
                                   apply_mask=True, boxes0=boxes)
    assert torch.equal(torch.isnan(got), torch.isnan(want))
    assert torch.equal(torch.nan_to_num(got), torch.nan_to_num(want))
    # level 1 as boxes too
    poison = torch.full((E, H * W, 16, 20), float("nan"), device=dev)
    del poison
    boxes1 = ops.build_boxes(planes[0], planes[1], ii, jj, coords, level=1)
    c1 = torch.nan_to_num(coords.reshape(E, H * W, 2), nan=0.0) * 0.5
    fx1 = torch.floor(c1[..., 0]).clamp(-64, W // 2 + 64).long()
    fy1 = torch.floor(c1[..., 1]).clamp(-64, H // 2 + 64).long()
    X1 = (((fx1 - 7) >> 2) << 2)[..., None, None] + torch.arange(20, device=dev).view(1, 1, 1, 20)
    Y1 = (fy1 - 7)[..., None, None] + torch.arange(16, device=dev).view(1, 1, 16, 1)
    ok1 = (X1 >= 0) & (X1 < W // 2) & (Y1 >= 0) & (Y1 < H // 2)
    idx1 = (Y1.clamp(0, H // 2 - 1) * (W // 2) + X1.clamp(0, W // 2 - 1)).reshape(E, H * W, 320)
    want1 = torch.where(ok1.reshape(E, H * W, 320), dense[1].reshape(E, H * W, H * W // 4).gather(2, idx1),
                        torch.zeros((), device=dev)).view(E, H * W, 16, 20)
    assert torch.equal(boxes1, want1)
    got2 = ops.altcorr_lookup_fused([None, None] + dense[2:], coords, off[0], off[1].clone(), 3, shared_offsets=False,
                                    apply_mask=True, boxes0=boxes, boxes1=boxes1)
    assert torch.equal(torch.isnan(got2), torch.isnan(want))
    assert torch.equal(torch.nan_to_num(got2), torch.nan_to_num(want))
    out16 = torch.zeros(E, 196, H, W, dtype=torch.float16, device=dev)
    ops.altcorr_lookup_fused([None] + dense[1:], coords, off[0], off[1].clone(), 3, shared_offsets=False, apply_mask=True,
                             boxes0=boxes, out=out16)
    assert torch.equal(torch.nan_to_num(out16.float()), torch.nan_to_num(want.half().float()))

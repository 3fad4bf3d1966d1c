"""GPU tests against the REFERENCE ITSELF: the original project's CUDA kernels recompiled, unmodified, for sm_100.

Two things are pinned here:
  1. the CPU oracle (oracle/lgu_oracle.c) == the reference kernels          -> "the oracle is right";
  2. the sm_100a product kernels (through the C ABI) == the reference kernels -> the drop-in claim.
The reference's outputs come from three places:
  - the reference modules themselves (oracle/_ref, built by oracle/build_ref.py from the original sources, which this
    repository does not contain), where they are built;
  - otherwise StoredReference below: the same operators for the cases of this file, checked against SHA-256
    fingerprints of the reference's outputs (tests/golden/ref_fingerprints.json);
  - tests/golden/ref_golden.pt: the reference's outputs themselves for small seeded cases (tests/golden/make_golden.py),
    against which the product kernels are checked at the end of this file (the oracle, on the CPU, in
    tests/test_golden_cpu.py)."""
import hashlib
import json
import os

import pytest
import torch

import inputs

pytestmark = pytest.mark.gpu
ATOL = 1e-5
HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden", "ref_golden.pt")
FINGERPRINTS = os.path.join(HERE, "golden", "ref_fingerprints.json")
# set to a path to write the fingerprints of StoredReference's results there instead of checking them
RECORD = os.environ.get("LGU_RECORD_REF_FINGERPRINTS")


def fingerprint(t):
    """SHA-256 of a tensor under eq_nan's equality: the NaN positions, then the values with NaN -> 0 and -0.0 -> +0.0."""
    t = t.detach().float().cpu().contiguous()
    h = hashlib.sha256(torch.isnan(t).numpy().tobytes())
    h.update((torch.nan_to_num(t, nan=0.0) + 0.0).numpy().tobytes())
    return h.hexdigest()


def _host(t):
    return t.detach().cpu().contiguous()


class StoredReference:
    """The reference modules' operators for the cases of this file, where the modules are not built.

    With the modules built, these tests found the CPU oracle bit-identical to the reference on exactly these inputs for
    the four lookups (outputs and in-place offset edits), and the product kernel bit-identical for gaussianMask.  So a
    call here computes its result with that implementation and checks it against the stored SHA-256 of the reference's
    output before returning it: a change in either is caught as a departure from the reference.
    gaussianMask_backward, lowMem_defSample and altcorr_forward matched the reference within 1e-5, not bit for bit, so
    no fingerprint of the reference's values exists for them: they return the oracle's values (the offset edits of
    lowMem_defSample are still checked)."""

    def __init__(self, oracle, ops, table):
        self.orc, self.ops, self.table = oracle, ops, table

    def _run(self, op, args, exact, impl, offset=None):
        key = op + ":" + ",".join(fingerprint(a) if torch.is_tensor(a) else repr(a) for a in args)
        host_off = _host(offset).clone() if offset is not None else None
        outs = impl(host_off)
        if offset is not None:
            offset.copy_(host_off)
        got = ([fingerprint(t) for t in outs] if exact else []) + ([fingerprint(host_off)] if offset is not None else [])
        if RECORD:
            self.table[key] = got
        else:
            assert key in self.table, f"no stored reference output for this {op} case"
            assert got == self.table[key], f"{op}: result differs from the reference's stored output"
        return [t.to(args[0].device) for t in outs]

    def corr_index_forward(self, vol, coords, r):
        return self._run("corr_index_forward", (vol, coords, r), True,
                         lambda _: self.orc.corr_index_forward(_host(vol), _host(coords), r))

    def corr_index_backward(self, vol, coords, grad, r):
        return self._run("corr_index_backward", (vol, coords, grad, r), True,
                         lambda _: self.orc.corr_index_backward(_host(vol), _host(coords), _host(grad), r))

    def defCorr_index_forward(self, vol, coords, off, r):
        return self._run("defCorr_index_forward", (vol, coords, off, r), True,
                         lambda o: self.orc.defCorr_index_forward(_host(vol), _host(coords), o, r), off)

    def defCorr_index_backward(self, vol, coords, off, grad, r):
        return self._run("defCorr_index_backward", (vol, coords, off, grad, r), True,
                         lambda o: self.orc.defCorr_index_backward(_host(vol), _host(coords), o, _host(grad), r), off)

    def gaussianMask(self, m, cv, vol, r):
        return self._run("gaussianMask", (m, cv, vol, r), True, lambda _: self.ops.gaussianMask(m, cv, vol, r))

    def gaussianMask_backward(self, m, cv, vol, g, r):
        return self._run("gaussianMask_backward", (m, cv, vol, g, r), False,
                         lambda _: self.orc.gaussianMask_backward(_host(m), _host(cv), _host(vol), _host(g), r))

    def lowMem_defSample(self, f1, f2, coords, off, r):
        return self._run("lowMem_defSample", (f1, f2, coords, off, r), False,
                         lambda o: self.orc.lowMem_defSample(_host(f1), _host(f2), _host(coords), o, r, strict_ref=True),
                         off)

    def altcorr_forward(self, f1, f2, coords, r):
        return self._run("altcorr_forward", (f1, f2, coords, r), False,
                         lambda _: self.orc.altcorr_forward(_host(f1), _host(f2), _host(coords), r))


@pytest.fixture(scope="module")
def gold():
    return torch.load(GOLD, weights_only=False)


@pytest.fixture(scope="module")
def stored_ref(oracle):
    import lgu_slam_b200
    table = {}
    if not RECORD:
        with open(FINGERPRINTS) as f:
            table = json.load(f)
    yield StoredReference(oracle, lgu_slam_b200.ops, table)
    if RECORD:
        with open(RECORD, "w") as f:
            json.dump(table, f, indent=1, sort_keys=True)


@pytest.fixture(scope="module")
def ref(stored_ref):
    from oracle import build_ref
    return build_ref.load_ref("defCorrSample_ref") or stored_ref


@pytest.fixture(scope="module")
def ref_alt(stored_ref):
    from oracle import build_ref
    return build_ref.load_ref("altcorr_ref") or stored_ref


def cu(t):
    return t.cuda().contiguous()


def eq_nan(a, b):
    return torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(torch.nan_to_num(a), torch.nan_to_num(b))


SHAPES = [(2, 6, 8, 6, 8, 3, True), (1, 48, 64, 48, 64, 3, True), (2, 48, 64, 24, 32, 3, True),
          (2, 48, 64, 12, 16, 3, False), (2, 48, 64, 6, 8, 3, True), (2, 48, 64, 24, 32, 1, True),
          (1, 5, 7, 9, 11, 2, True), (1, 20, 20, 6, 6, 4, False)]


@pytest.mark.parametrize("E,H1,W1,H2,W2,r,probes", SHAPES)
def test_forward_lookups_bit_exact_vs_reference(ops, oracle, ref, E, H1, W1, H2, W2, r, probes):
    c = inputs.volume_case(E, H1, W1, H2, W2, r, seed=1000 + r, probes=probes)
    vol, coords = cu(c["volume"]), cu(c["coords"])
    # plain lookup
    want, = ref.corr_index_forward(vol, coords, r)
    got, = ops.corr_index_forward(vol, coords, r)
    orc, = oracle.corr_index_forward(c["volume"], c["coords"], r)
    assert eq_nan(got, want), "product corr_index_forward != reference (bit-exact expected)"
    assert eq_nan(orc, want.cpu()), "oracle corr_index_forward != reference (bit-exact expected)"
    # deformable lookup + in-place offset mutation
    o_ref, o_got, o_orc = cu(c["offset"]), cu(c["offset"]), c["offset"].clone()
    want, = ref.defCorr_index_forward(vol, coords, o_ref, r)
    got, = ops.defCorr_index_forward(vol, coords, o_got, r)
    orc, = oracle.defCorr_index_forward(c["volume"], c["coords"], o_orc, r)
    assert eq_nan(got, want) and torch.equal(o_got, o_ref)
    assert eq_nan(orc, want.cpu()) and torch.equal(o_orc, o_ref.cpu())


@pytest.mark.parametrize("E,H1,W1,H2,W2,r,probes", SHAPES)
def test_backward_lookups_vs_reference(ops, oracle, ref, E, H1, W1, H2, W2, r, probes):
    c = inputs.volume_case(E, H1, W1, H2, W2, r, seed=1100 + r, probes=probes)
    vol, coords, grad = cu(c["volume"]), cu(c["coords"]), cu(c["corr_grad"])
    want, = ref.corr_index_backward(vol, coords, grad, r)
    got, = ops.corr_index_backward(vol, coords, grad, r)
    orc, = oracle.corr_index_backward(c["volume"], c["coords"], c["corr_grad"], r)
    assert torch.allclose(got, want, atol=ATOL, rtol=0, equal_nan=True)
    assert eq_nan(orc, want.cpu()), "oracle follows the reference's accumulation order: bit-exact expected"
    o_ref, o_got, o_orc = cu(c["offset"]), cu(c["offset"]), c["offset"].clone()
    wv, wo = ref.defCorr_index_backward(vol, coords, o_ref, grad, r)
    gv, go = ops.defCorr_index_backward(vol, coords, o_got, grad, r)
    ov, oo = oracle.defCorr_index_backward(c["volume"], c["coords"], o_orc, c["corr_grad"], r)
    assert torch.allclose(gv, wv, atol=ATOL, rtol=0, equal_nan=True)
    assert eq_nan(go, wo), "offset_grad: same operation order as the reference -> bit-exact"
    assert torch.equal(o_got, o_ref)
    assert eq_nan(ov, wv.cpu()) and eq_nan(oo, wo.cpu()) and torch.equal(o_orc, o_ref.cpu())


@pytest.mark.parametrize("E,H1,W1,H2,W2,r,probes", [(2, 6, 8, 6, 8, 4, True), (1, 48, 64, 48, 64, 4, True),
                                                    (2, 5, 7, 9, 11, 4, True), (1, 4, 4, 10, 12, 2, False)])
def test_gaussian_vs_reference(ops, oracle, ref, E, H1, W1, H2, W2, r, probes):
    c = inputs.gaussian_case(E, H1, W1, H2, W2, r, seed=1200 + r, probes=probes)
    m, cv, vol, g = cu(c["means"]), cu(c["covs"]), cu(c["volume"]), cu(c["out_grad"])
    want, = ref.gaussianMask(m, cv, vol, r)
    got, = ops.gaussianMask(m, cv, vol, r)
    orc, = oracle.gaussianMask(c["means"], c["covs"], c["volume"], r)
    assert torch.equal(got, want), "same arithmetic + same CUDA expf -> bit-exact"
    assert torch.equal(orc == 0, want.cpu() == 0)
    assert torch.allclose(orc, want.cpu(), atol=ATOL, rtol=1e-6)          # glibc expf vs CUDA expf
    wm, wc = ref.gaussianMask_backward(m, cv, vol, g, r)
    gm, gc = ops.gaussianMask_backward(m, cv, vol, g, r)
    om, oc = oracle.gaussianMask_backward(c["means"], c["covs"], c["volume"], c["out_grad"], r)
    for a, b in ((gm, wm), (gc, wc), (om.cuda(), wm), (oc.cuda(), wc)):
        assert torch.allclose(a, b, atol=ATOL, rtol=1e-5), (a - b).abs().max()


@pytest.mark.parametrize("B,N,H1,W1,H2,W2,C,r,probes", [(3, 1, 6, 8, 6, 8, 128, 3, True),
                                                        (2, 1, 48, 64, 48, 64, 128, 3, True),
                                                        (2, 1, 48, 64, 12, 16, 128, 3, False),
                                                        (2, 2, 5, 7, 4, 6, 64, 2, True)])
def test_lowmem_vs_reference(ops, oracle, ref, B, N, H1, W1, H2, W2, C, r, probes):
    c = inputs.lowmem_case(B, N, H1, W1, H2, W2, C, r, seed=1300 + r, probes=probes)
    f1, f2, coords = cu(c["fmap1"]), cu(c["fmap2"]), cu(c["coords"])
    o_ref, o_got, o_orc = cu(c["offset"]), cu(c["offset"]), c["offset"].clone()
    want, = ref.lowMem_defSample(f1, f2, coords, o_ref, r)                 # the reference IS strict (quirk Q2)
    got, = ops.lowMem_defSample(f1, f2, coords, o_got, r, strict_ref=True)
    orc, = oracle.lowMem_defSample(c["fmap1"], c["fmap2"], c["coords"], o_orc, r, strict_ref=True)
    assert torch.allclose(got, want, atol=ATOL, rtol=0, equal_nan=True), (got - want).abs().nan_to_num().max()
    assert torch.allclose(orc, want.cpu(), atol=ATOL, rtol=0, equal_nan=True)
    assert torch.equal(o_got, o_ref) and torch.equal(o_orc, o_ref.cpu())


@pytest.mark.parametrize("B,N,H1,W1,H2,W2,C,r,probes", [(3, 1, 6, 8, 6, 8, 128, 1, True),
                                                        (2, 1, 48, 64, 24, 32, 128, 1, True),
                                                        (2, 2, 5, 7, 4, 6, 64, 3, True)])
def test_altcorr_vs_reference(ops, oracle, ref_alt, B, N, H1, W1, H2, W2, C, r, probes):
    c = inputs.lowmem_case(B, N, H1, W1, H2, W2, C, r, seed=1400 + r, probes=probes)
    f1, f2, coords = cu(c["fmap1"]), cu(c["fmap2"]), cu(c["coords"])
    want, = ref_alt.altcorr_forward(f1, f2, coords, r)
    got, = ops.altcorr_forward(f1, f2, coords, r)
    orc, = oracle.altcorr_forward(c["fmap1"], c["fmap2"], c["coords"], r)
    assert torch.allclose(got, want, atol=ATOL, rtol=0, equal_nan=True), (got - want).abs().nan_to_num().max()
    assert torch.allclose(orc, want.cpu(), atol=ATOL, rtol=0, equal_nan=True)


# ------------------------------------------------------------------------------------------------ stored reference outputs
@pytest.mark.parametrize("name", ["lvl_a", "lvl_b", "lvl_c"])
def test_lookup_kernels_vs_reference_golden(ops, gold, name):
    G = gold[name]
    c = inputs.volume_case(**G["kw"])
    r = G["kw"]["r"]
    vol, coords, grad = cu(c["volume"]), cu(c["coords"]), cu(c["corr_grad"])
    got, = ops.corr_index_forward(vol, coords, r)
    assert eq_nan(got.cpu(), G["corr_index_forward"]), "product corr_index_forward != reference (bit-exact expected)"
    o_got = cu(c["offset"])
    got, = ops.defCorr_index_forward(vol, coords, o_got, r)
    assert eq_nan(got.cpu(), G["defCorr_index_forward"]) and torch.equal(o_got.cpu(), G["offset_after"])
    got, = ops.corr_index_backward(vol, coords, grad, r)
    assert torch.allclose(got.cpu(), G["corr_index_backward"], atol=ATOL, rtol=0, equal_nan=True)
    gv, go = ops.defCorr_index_backward(vol, coords, cu(c["offset"]), grad, r)
    wv, wo = G["defCorr_index_backward"]
    assert torch.allclose(gv.cpu(), wv, atol=ATOL, rtol=0, equal_nan=True)
    assert eq_nan(go.cpu(), wo), "offset_grad: same operation order as the reference -> bit-exact"


@pytest.mark.parametrize("name", ["gauss_a", "gauss_b"])
def test_gaussian_kernels_vs_reference_golden(ops, gold, name):
    G = gold[name]
    c = inputs.gaussian_case(**G["kw"])
    r = G["kw"]["r"]
    m, cv, vol, g = cu(c["means"]), cu(c["covs"]), cu(c["volume"]), cu(c["out_grad"])
    got, = ops.gaussianMask(m, cv, vol, r)
    assert torch.equal(got.cpu(), G["gaussianMask"]), "same arithmetic + same CUDA expf -> bit-exact"
    gm, gc = ops.gaussianMask_backward(m, cv, vol, g, r)
    for a, b in ((gm, G["gaussianMask_backward"][0]), (gc, G["gaussianMask_backward"][1])):
        assert torch.allclose(a.cpu(), b, atol=ATOL, rtol=1e-5), (a.cpu() - b).abs().max()


@pytest.mark.parametrize("name", ["lowmem_a", "lowmem_b"])
def test_lowmem_altcorr_kernels_vs_reference_golden(ops, gold, name):
    G = gold[name]
    c = inputs.lowmem_case(**G["kw"])
    r = G["kw"]["r"]
    f1, f2, coords, o_got = cu(c["fmap1"]), cu(c["fmap2"]), cu(c["coords"]), cu(c["offset"])
    got, = ops.lowMem_defSample(f1, f2, coords, o_got, r, strict_ref=True)       # the reference IS strict (quirk Q2)
    assert torch.allclose(got.cpu(), G["lowMem_defSample"], atol=ATOL, rtol=0, equal_nan=True)
    assert torch.equal(o_got.cpu(), G["offset_after"])
    got, = ops.altcorr_forward(f1, f2, coords, r)
    assert torch.allclose(got.cpu(), G["altcorr_forward"], atol=ATOL, rtol=0, equal_nan=True)

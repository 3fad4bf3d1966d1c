"""The offset heads' glue in training (corr.py:117-135, per_Corr_Normalization :44-51), forward + backward, on one GPU.

  chain   what CorrBlock ran before the heads had a backward: the torch chain in autograd (mean, var, sqrt, sub, div, tanh,
          x4 per head, F.interpolate, add, /2, two permutes) plus the first fused lookup's .float().contiguous() copies of
          both permuted offset tensors, and autograd's backward of all of it
  fused   corr.OffsetHeads: lgu_offset_heads (2 launches) + lgu_offset_heads_backward (2 launches)

Both arms run alternately in one process on the same inputs (c0 [E,98,48,64], c1 [E,98,24,32] stand in for the conv
outputs; random upstream gradients on both offset tensors), timed with CUDA events.  The backward kernel pair is also timed
alone, and its rate is given on the algorithmic 1764 B per source pixel at CH = 98 (read G0, G1, c0, c1 once: 784 + 392
+ 98 B; write g_c0, g_c1: 392 + 98 B) against the 6552 GB/s copy peak measured for this project on a B200.  The working
set (>= 190 MB at E = 48) exceeds the 126 MB L2, so every pass reads HBM.

    python tools/bench_offset_heads.py [--edges 48,96] [--iters 50] [--warmup 5]

Prints one JSON line per edge count.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

COPY_PEAK_GBS = 6552.0
CH, H, W = 98, 48, 64


def bytes_per_pixel(ch=CH):
    return 4 * (2 * ch + ch) + ch + 4 * ch + ch                  # read G0, G1, c0 and c1 (ch / 4 per pixel); write g_c0, g_c1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--edges", default="48,96")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    assert bytes_per_pixel() == 1764

    import torch
    import torch.nn.functional as F
    import inputs
    import lgu_slam_b200  # noqa: F401
    from importlib import import_module
    corr = import_module("lgu-slam_b200.corr")
    ops = corr.ops
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing measured")
    dev = torch.device("cuda:0")

    def chain(c0, c1, g0, g1):
        o1 = F.interpolate(c1, (H, W))
        o0 = torch.tanh(corr.per_Corr_Normalization(c0, [1, 2, 3])) * 4
        o1 = (torch.tanh(corr.per_Corr_Normalization(o1, [1, 2, 3])) * 4 + o0) / 2
        r0 = o0.permute(0, 2, 3, 1).float().contiguous()
        r1 = o1.permute(0, 2, 3, 1).float().contiguous()
        torch.autograd.backward([r0, r1], [g0, g1])

    def fused(c0, c1, g0, g1):
        r0, r1 = corr.OffsetHeads.apply(c0, c1)
        torch.autograd.backward([r0, r1], [g0, g1])

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / n                      # us per call

    for E in [int(x) for x in a.edges.split(",")]:
        g = inputs.gen(1000 + E)
        c0 = (torch.randn(E, CH, H, W, generator=g) * 1.7 + 0.3).to(dev).requires_grad_()
        c1 = (torch.randn(E, CH, H // 2, W // 2, generator=g) * 0.6 - 0.2).to(dev).requires_grad_()
        g0 = torch.randn(E, H, W, CH, generator=g).to(dev)
        g1 = torch.randn(E, H, W, CH, generator=g).to(dev)
        arms = {"chain": lambda: chain(c0, c1, g0, g1), "fused": lambda: fused(c0, c1, g0, g1)}
        grads = {}
        for name, fn in arms.items():
            c0.grad = c1.grad = None
            fn()
            grads[name] = (c0.grad.clone(), c1.grad.clone())
        err = max((grads["fused"][k] - grads["chain"][k]).abs().max().item() for k in range(2))
        ts = {k: [] for k in arms}
        for _ in range(a.warmup):
            for fn in arms.values():
                fn()
        for _ in range(a.iters):                                   # alternate the arms, one call each
            for name, fn in arms.items():
                c0.grad = c1.grad = None
                ts[name].append(timed(fn, 1))
        c0d, c1d = c0.detach(), c1.detach()
        _, _, stats = ops.offset_heads(c0d, c1d, return_stats=True)
        bwd = lambda: ops.offset_heads_backward(c0d, c1d, stats, g0, g1)
        fwd = lambda: ops.offset_heads(c0d, c1d)
        for _ in range(a.warmup):
            bwd(); fwd()
        t_bwd = timed(bwd, a.iters)
        t_fwd = timed(fwd, a.iters)
        nbytes = bytes_per_pixel() * E * H * W
        gbs = nbytes / (t_bwd * 1e-6) / 1e9
        print(json.dumps({
            "edges": E, "grid": [H, W], "channels": CH,
            "chain_us": round(statistics.median(ts["chain"]), 1),
            "fused_us": round(statistics.median(ts["fused"]), 1),
            "chain_us_spread": [round(min(ts["chain"]), 1), round(max(ts["chain"]), 1)],
            "fused_us_spread": [round(min(ts["fused"]), 1), round(max(ts["fused"]), 1)],
            "fwd_kernels_us": round(t_fwd, 1), "bwd_kernels_us": round(t_bwd, 1),
            "bwd_algorithmic_MB": round(nbytes / 1e6, 1), "bwd_GB_per_s_on_1764B_per_px": round(gbs, 1),
            "bwd_fraction_of_copy_peak": round(gbs / COPY_PEAK_GBS, 3),
            "max_grad_diff_fused_vs_chain": err,
            "device": torch.cuda.get_device_name(dev)}), flush=True)
        del c0, c1, g0, g1, grads, c0d, c1d, stats
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

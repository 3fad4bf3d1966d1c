"""BASELINE configs[2]: the train.py step shape through the correlation path, forward AND backward, on one B200.

A training step of the reference (droid_net.py:187-222, train.py:119-122,202-216) builds ONE CorrBlock for the clip's
edges (batch b x n edges per clip) and looks it up `num_steps` times; `loss.backward()` then runs every lookup's backward
(4 x defCorr_index_backward + corr_index_backward, each zero-filling a dense volume_grad), sums those dense gradients
and goes back through avg_pool2d / gaussianMask / matmul.  This tool times exactly that slice -- CorrBlock.__init__,
num_steps x CorrBlock.__call__, backward to the feature maps and the offset / Gaussian heads -- in four arms:

  acc      this repo, fused build + fused lookups, level gradients accumulated in persistent buffers (the default)
  dense    this repo, fused build + fused lookups, one dense gradient per lookup summed by autograd
  per_op   this repo's drop-in operators inside the reference's per-operator graph (fused=False)
  acc_chain  `acc` with the offset heads' torch chain patched back in (permuted views, autograd backward): the same-process
           comparison for corr.OffsetHeads
  acc_conv `acc` with corr.OffsetConv heads (the same parameters): the offset convolutions on the library's tensor-core
           kernels instead of cuDNN fp32
  ref_cuda the reference's OWN kernels recompiled unmodified for sm_100 (oracle/_ref) inside the same per-operator
           graph (skipped when oracle/_ref is absent)

    python tools/bench_train.py [--batch 4] [--edges 24] [--steps 9] [--iters 3] [--arms acc,dense,per_op,acc_chain,acc_conv,ref_cuda]

Prints one JSON line per arm (CUDA events around whole training steps, median).  Inputs are synthetic (fp32 maps, as
in training), TF32 off.  The conv heads (ofsMap / ofs_residual, cuDNN fp32) are part of every arm alike, except acc_conv.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--edges", type=int, default=24, help="edges per clip (train.py --edges)")
    ap.add_argument("--steps", type=int, default=9, help="lookups per training step (train.py --iters / num_steps)")
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--arms", default="per_op,acc,dense,ref_cuda")
    a = ap.parse_args()

    import torch
    import torch.nn as nn
    import inputs
    import lgu_slam_b200
    from importlib import import_module
    corr = import_module("lgu-slam_b200.corr")
    dev = torch.device("cuda:0")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    H, W, C = 48, 64, 128
    b, n = a.batch, a.edges
    E = b * n
    g = inputs.gen(1234 + 3)
    fm1 = torch.randn(b, n, C, H, W, generator=g).to(dev)
    fm2 = torch.randn(b, n, C, H, W, generator=g).to(dev)
    coords = [inputs.make_coords(E, H, W, H, W, g).permute(0, 2, 3, 1).contiguous().view(b, n, H, W, 2).to(dev)
              for _ in range(a.steps)]
    wts = [torch.randn(b, n, 196, H, W, generator=g).to(dev) for _ in range(a.steps)]
    torch.manual_seed(7)
    ofsMap = nn.Conv2d(256, 98, 3, padding=1).to(dev)
    ofs_residual = nn.Conv2d(256, 98, 3, padding=1).to(dev)
    GA = corr.GaussianMask(H, W).to(dev)
    conv_heads = [corr.OffsetConv(256, 98).to(dev) for _ in range(2)]
    for h, ref_h in zip(conv_heads, (ofsMap, ofs_residual)):
        h.load_state_dict(ref_h.state_dict())
    params = [p for m in (ofsMap, ofs_residual, GA, *conv_heads) for p in m.parameters()]

    real_ops = corr.ops
    real_offsets = corr._generate_offsets

    def train_step(kind):
        f1, f2 = fm1.clone().requires_grad_(), fm2.clone().requires_grad_()
        for p in params:
            p.grad = None
        fused = kind in ("acc", "dense", "acc_chain", "acc_conv")
        heads = conv_heads if kind == "acc_conv" else (ofsMap, ofs_residual)
        blk = corr.CorrBlock(*heads, GA, f1, f2, fused=fused, fused_lookup=fused,
                             accumulate_grads=(kind in ("acc", "acc_chain", "acc_conv")))
        loss = 0.0
        for c, w in zip(coords, wts):
            out, mean_n, theta = blk(c)
            loss = loss + (out * w).mean() + 1e-3 * (mean_n.square().mean() + theta.mean())
        loss.backward()
        return f1.grad, f2.grad

    results = {}
    for kind in a.arms.split(","):
        if kind == "ref_cuda":
            from oracle import build_ref
            ref = build_ref.load_ref("defCorrSample_ref")
            if ref is None:
                print(json.dumps({"arm": kind, "unavailable": "oracle/_ref/defCorrSample_ref.so is absent"}))
                continue
            corr.ops = ref                                   # the 6 operator names CorrBlock's per-op graph calls
        if kind == "acc_chain":
            corr._generate_offsets = lambda ofsMap, ofs_residual, t, fused_lookup=False: real_offsets(ofsMap, ofs_residual, t)
        try:
            torch.cuda.reset_peak_memory_stats()
            g1, _ = train_step(kind)
            torch.cuda.synchronize()
            ts = []
            for _ in range(a.iters):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                train_step(kind)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            ms = statistics.median(ts)
            results[kind] = g1.detach().clone()
            line = {"arm": kind, "ms_per_train_step": round(ms, 3), "edges": E, "lookups_per_step": a.steps,
                    "edge_lookups_fwd_bwd_per_s": round(E * a.steps / (ms * 1e-3), 1),
                    "peak_mem_GB": round(torch.cuda.max_memory_allocated() / 2**30, 2),
                    "fmap1_grad_rms": float(g1.square().mean().sqrt())}
            if "per_op" in results and kind != "per_op":
                line["fmap1_grad_max_err_vs_per_op"] = float((g1 - results["per_op"]).abs().max())
            if kind == "acc_conv" and "acc" in results:
                line["fmap1_grad_max_err_vs_acc"] = float((g1 - results["acc"]).abs().max())
            print(json.dumps(line), flush=True)
        finally:
            corr.ops = real_ops
            corr._generate_offsets = real_offsets
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
